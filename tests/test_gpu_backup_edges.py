"""
Every backup path against the extended-precision reference (oracle/highprec.py) at its tile, slab and dispatch boundaries.

The contract is `highprec.check_backup`: v* and a* are the exact argmax wherever the exact gap exceeds twice the certified bound of
any float64 evaluation order; values are within that bound of the exact value at the engine's own v*; rows are bitwise the float64
restatement of alpha_a_entry.  Where a path is otherwise invisible (slab loops, grouped vs plain assemble, Gamma z-groups) the launch
count of the call (`pbvi_last_launches`) shows that the path was taken.
"""
import ctypes
import itertools

import numpy as np
import pytest

from conftest import load_golden
from oracle import highprec as hp
from oracle import pbvi_oracle as orc

pytestmark = pytest.mark.gpu

GAMMA = 0.95
GRID_Y = 65535                     # CUDA grid.y limit: the slab size of the value pass, the plain assemble kernel and GER
ASM_G = 8                          # tuples per block of the grouped assemble kernel (PBVI_ASM_G in backup.cu)


@pytest.fixture(scope='module')
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), 'these tests need a CUDA device'
    return torch


# ---- models and inputs ---------------------------------------------------------------------------------------------------------
def synthetic(S, A, O, R, seed, negative=False, landing=None):
    """configs[4] recipe with non-uniform transition probabilities: random landing states (drawn from `landing` when given),
    impossible observations, reward 1 on reaching S // 2; `negative` subtracts a random penalty from the expected rewards."""
    rng = np.random.default_rng(seed)
    reach = rng.integers(0, S, (S, A, R)) if landing is None else rng.choice(landing, (S, A, R))
    probs = rng.random((S, A, R)) + 0.05
    probs /= probs.sum(2, keepdims=True)
    obs = rng.random((S, A, O))
    obs /= obs.sum(2, keepdims=True)
    obs[rng.random((S, A, O)) < 0.3] = 0.0
    rto = orc.build_rto(reach, probs, obs)
    rbar = orc.expected_rewards(rto, orc.end_state_reachable_rewards(reach, O, [S // 2]))
    if negative:
        rbar = rbar - 0.3 * rng.random((S, A))
    return reach, probs, rto, rbar


def sparse_beliefs(rng, n, S, ks):
    B = np.zeros((n, S))
    for i in range(n):
        k = min(S, ks[i % len(ks)])
        idx = rng.choice(S, k, replace=False)
        B[i, idx] = rng.dirichlet(np.ones(k))
    return B


def alphas_for(rng, nV, S, negative):
    V = rng.random((nV, S))
    return 2.0 * V - 1.0 if negative else V


def device(model):
    from pomdp_pbvi_exploration_b200._native import DeviceModel
    reach, probs, rto, rbar = model
    return DeviceModel(reach, probs, rto, rbar)


def launches(dev):
    return dev._lib.pbvi_last_launches(dev._h)


def backup_checked(dev, model, B, V, gamma=GAMMA):
    """pbvi_backup on (B, V) with the whole contract applied; returns the engine outputs as NumPy arrays."""
    reach, _, rto, rbar = model
    rows, act, vstar, value = [t.cpu().numpy() for t in dev.backup(B, V, gamma)]
    hp.check_backup(reach, rto, rbar, gamma, B, V, vstar, value, act, rows)
    return rows, act, vstar, value


def exact_decisions(model, B, V, gamma=GAMMA):
    """(v*, a*) of the exact backup; the inputs must leave every choice decided (or every term of a score row zero)."""
    reach, _, rto, rbar = model
    ex, bd, zero = hp.scores(reach, rto, B, V)
    vstar = np.argmax(ex, axis=3)
    flat = np.all(zero, axis=3)
    vstar[flat] = 0
    assert np.all(hp.check_argmax(ex, bd, vstar, zero) | flat), 'test inputs with an undecided v*'
    ev, evb = hp.values(reach, rto, rbar, gamma, B, V, vstar)
    astar = np.argmax(ev, axis=1)
    assert np.all(hp.check_argmax(ev, evb, astar)), 'test inputs with an undecided a*'
    return vstar, astar


def pairwise(factors, cost):
    """A small set of rows of the product of `factors` that holds every pair of values of every two factors (greedy, cheapest first)."""
    pairs = list(itertools.combinations(range(len(factors)), 2))
    todo = {(i, x, j, y) for i, j in pairs for x in factors[i] for y in factors[j]}
    cands = sorted(itertools.product(*factors), key=cost)
    rows = []
    while todo:
        best = max(cands, key=lambda c: sum((i, c[i], j, c[j]) in todo for i, j in pairs))
        rows.append(best)
        todo -= {(i, best[i], j, best[j]) for i, j in pairs}
    return rows


# ---- tile edges ------------------------------------------------------------------------------------------------------------------
# S crosses the 4-state chunk, the 16-chunk stage and BN; nV the 64-column quarter, the 256-column tile and columns beyond V; nB the
# 16-row group and the 64-row tile.
TILE_CASES = pairwise([(1, 2, 17, 255, 257, 1023), (1, 63, 64, 65, 255, 256, 257, 513), (1, 15, 16, 17, 63, 64, 65), (1, 2, 3)],
                      cost=lambda c: c[0] * c[1] * c[2] * c[3])


@pytest.mark.parametrize('S,nV,nB,R', TILE_CASES)
def test_tile_edges(torch_cuda, S, nV, nB, R):
    negative = (S + nV + nB) % 2 == 1
    model = synthetic(S, 2, 3, R, seed=S * 1000 + nV * 10 + R, negative=negative)
    rng = np.random.default_rng(nB * 7 + S)
    B = sparse_beliefs(rng, nB, S, [min(S, 257), 40, 5, 1])
    V = alphas_for(rng, nV, S, negative)
    dev = device(model)
    backup_checked(dev, model, B, V)
    dev.close()


# ---- dispatch shapes -------------------------------------------------------------------------------------------------------------
DISPATCH = [  # A, O, R, negative rewards
    (1, 1, 1, False), (2, 2, 1, True), (5, 3, 1, False), (9, 4, 1, True), (2, 5, 1, False), (5, 8, 1, True), (9, 8, 1, False),
    (9, 1, 2, True), (1, 2, 3, False), (2, 3, 2, True), (5, 4, 2, False), (9, 5, 2, False), (2, 8, 3, True), (1, 5, 2, True),
]


@pytest.mark.parametrize('A,O,R,negative', DISPATCH)
def test_dispatch_shapes(torch_cuda, A, O, R, negative):
    """Every action / observation count of the score and assemble dispatch (grouped assemble templates OM = 2 / 3 / 4, the plain
    kernel for O >= 5 or R > 1), with and without negative rewards (only non-negative models reach the value pass's screening and its
    exact-zero shortcut)."""
    S, nB, nV = 200, 70, 70
    model = synthetic(S, A, O, R, seed=A * 100 + O * 10 + R, negative=negative)
    rng = np.random.default_rng(A + O + R)
    B = sparse_beliefs(rng, nB, S, [S, 40, 5, 1])
    B[::9] = 0.0
    B[::9, :4] = 0.25                                         # a few beliefs on one corner chunk: exact-zero scores for some (a, o)
    V = alphas_for(rng, nV, S, negative)
    dev = device(model)
    rows, act, vstar, _ = backup_checked(dev, model, B, V)
    # assemble of the selected tuples: the grouped kernel (one scan + order + grouped launch) or the plain one (scan + one slab)
    sel = vstar[np.arange(nB), act]
    again = dev.backup_assemble(V, GAMMA, act, sel).cpu().numpy()
    grouped = R == 1 and O <= 4 and nB >= 4 * ASM_G
    assert launches(dev) == (3 if grouped else 2)
    assert again.tobytes() == rows.tobytes()
    dev.close()


@pytest.mark.parametrize('S,R', [(1, 1), (2, 1), (2, 2)])
@pytest.mark.parametrize('nB', [64, 65])
def test_degenerate_shapes(torch_cuda, S, R, nB):
    """One action, one or two states, one alpha vector."""
    model = synthetic(S, 1, 2, R, seed=S + R)
    rng = np.random.default_rng(nB)
    B = rng.dirichlet(np.ones(S), size=nB)
    V = rng.random((1, S))
    dev = device(model)
    backup_checked(dev, model, B, V)
    dev.close()


# ---- adversarial content ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('R', [1, 2])
def test_duplicated_winner_lower_index_wins(torch_cuda, R):
    """The winning alpha repeated in its own column quarter, in another quarter and in another tile: bitwise identical columns give
    bitwise identical scores, and the lowest index must win (np.argmax)."""
    S, nB, nV = 300, 50, 600
    model = synthetic(S, 3, 3, R, seed=41 + R)
    rng = np.random.default_rng(43)
    B = sparse_beliefs(rng, nB, S, [S, 40, 5])
    V = rng.random((nV, S))
    V[5] += 1.0
    copies = [40, 70, 300]                                    # same quarter, next quarter, second alpha tile
    V[copies] = V[5]
    dev = device(model)
    rows, act, vstar, value = backup_checked(dev, model, B, V)
    assert not np.isin(vstar, copies).any()
    assert np.mean(vstar == 5) > 0.5
    _, arg = dev.max_values(B, V)
    assert not np.isin(arg.cpu().numpy(), copies).any()
    dev.close()


def test_alphas_a_few_ulps_apart(torch_cuda):
    S, nB, nV = 120, 40, 70
    model = synthetic(S, 2, 3, 1, seed=7)
    rng = np.random.default_rng(8)
    B = sparse_beliefs(rng, nB, S, [S, 40, 5, 1])
    V = rng.random((nV, S))
    base = V[3] + 1.0
    for i, v in enumerate(range(0, nV, 7)):                   # every 7th alpha: the same vector moved by i ulps, in both directions
        V[v] = base
        for _ in range(i):
            V[v] = np.nextafter(V[v], np.inf if i % 2 else -np.inf)
    dev = device(model)
    backup_checked(dev, model, B, V)
    dev.close()


@pytest.mark.parametrize('negative', [False, True])
def test_tiny_belief_entries_alone_in_a_chunk(torch_cuda, negative):
    """Belief entries of 1e-13 and 1e-310 that are the only non-zero entry of their 4-state chunk in their whole row group: a kernel
    that skips such a chunk drops a real term.  1e-13 of an O(1) entry is ~40 certified bounds; a belief made of 1e-310 entries only
    has subnormal scores whose gaps are still far above the bound."""
    S, nB = 1024, 64
    model = synthetic(S, 2, 3, 1, seed=11, negative=negative)
    rng = np.random.default_rng(12)
    B = np.zeros((nB, S))
    for b in range(nB):
        if b % 2 == 0:
            B[b, b % 4] = 1.0 - 1e-13                         # every belief shares chunk 0 ...
            B[b, 4 * (10 + b)] = 1e-13                        # ... and owns chunk 10 + b alone
        else:
            B[b, 4 * (100 + b) + 1] = 1e-310
            B[b, 4 * (180 + b) + 2] = 3e-310
    V = alphas_for(rng, 90, S, negative) + (0.0 if negative else 0.5)
    dev = device(model)
    backup_checked(dev, model, B, V)
    dev.close()


@pytest.mark.parametrize('R', [1, 2])
def test_alphas_zero_on_whole_tiles_mixed_signs(torch_cuda, R):
    S, nB, nV = 400, 70, 600
    model = synthetic(S, 3, 2, R, seed=21 + R)
    rng = np.random.default_rng(22)
    B = sparse_beliefs(rng, nB, S, [S, 40, 5, 1])
    V = 2.0 * rng.random((nV, S)) - 1.0
    V[256:512] = 0.0                                          # the whole second alpha tile
    V[:256, :200] = 0.0                                       # the first tile on every chunk of the first half of the states
    V[512:, rng.random(S) < 0.5] = 0.0
    dev = device(model)
    backup_checked(dev, model, B, V)
    dev.close()


# ---- launch-limit slabs ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def slab_case(torch_cuda):
    model = synthetic(8, 2, 2, 1, seed=3)
    rng = np.random.default_rng(4)
    nB = GRID_Y + 100
    B = rng.dirichlet(np.ones(8), size=nB)
    B[::3, :3] = 0.0
    B /= B.sum(1, keepdims=True)
    V = rng.random((5, 8))
    dev = device(model)
    yield model, dev, B, V
    dev.close()


def test_backup_and_select_walk_belief_slabs(slab_case):
    """nB = 65 535 + 100: the value pass and the assemble kernel each take a second slab; every output is checked, and the second
    slab's outputs equal a separate call on those beliefs."""
    model, dev, B, V = slab_case
    reach, _, rto, rbar = model
    rows, act, vstar, value = backup_checked(dev, model, B, V)
    n_big = launches(dev)
    dev.backup(B[:GRID_Y], V, GAMMA)
    assert n_big == launches(dev) + 2                         # one more value-pass slab, one more assemble slab
    tail = [t.cpu().numpy() for t in dev.backup(B[GRID_Y:], V, GAMMA)]
    for got, want in zip(tail, (rows, act, vstar, value)):
        assert got.tobytes() == want[GRID_Y:].tobytes()
    vs2, val2, as2 = [t.cpu().numpy() for t in dev.backup_select(B, V, GAMMA)]
    assert vs2.tobytes() == vstar.tobytes() and val2.tobytes() == value.tobytes() and as2.tobytes() == act.tobytes()
    # without the values: a* comes from the screened pass, which skips the exact sum when one action is the only contender
    vs3, _, as3 = [t.cpu().numpy() if t is not None else None for t in dev.backup_select(B, V, GAMMA, want_value=False)]
    assert vs3.tobytes() == vstar.tobytes()
    ev, evb = hp.values(reach, rto, rbar, GAMMA, B, V, vs3)
    hp.check_argmax(ev, evb, as3, what='a* (no values)')


def test_max_values_beyond_65535_beliefs(slab_case):
    model, dev, B, V = slab_case
    mx, arg = [t.cpu().numpy() for t in dev.max_values(B, V)]
    ex, bd, zero = hp.plain_scores(B, V)
    hp.check_argmax(ex, bd, arg, zero, what='max_values')
    hp.check_close(mx, np.take_along_axis(ex, arg[:, None].astype(np.int64), 1)[:, 0],
                   np.take_along_axis(bd, arg[:, None].astype(np.int64), 1)[:, 0], what='max_values')


def grouped_assemble_limit(A, G=ASM_G):
    """Largest tuple count the grouped assemble kernel takes: assemble_impl requires (n + A (G - 1)) / G + 1 <= 65535 (grid.y)."""
    n = GRID_Y * G - 1 - A * (G - 1)
    assert (n + A * (G - 1)) // G + 1 <= GRID_Y < (n + 1 + A * (G - 1)) // G + 1
    return n


@pytest.mark.parametrize('side', ['below', 'above'])
def test_assemble_around_the_grouped_kernel_limit(torch_cuda, side):
    S, A, O = 4, 2, 2
    model = synthetic(S, A, O, 1, seed=5)
    reach, _, rto, rbar = model
    n = grouped_assemble_limit(A) + (0 if side == 'below' else 1)
    rng = np.random.default_rng(6)
    V = rng.random((9, S))
    act = rng.integers(0, A, n).astype(np.int32)
    vsel = rng.integers(0, 9, (n, O)).astype(np.int32)
    dev = device(model)
    rows, keys = dev.backup_assemble(V, GAMMA, act, vsel, with_hash=True)
    # grouped: scan + order + grouped kernel + hash finalise; plain: scan + one launch per 65 535 tuples + hash finalise
    assert launches(dev) == (4 if side == 'below' else 2 + -(-n // GRID_Y))
    assert torch_cuda.equal(keys, dev.row_hash(rows))
    assert rows.cpu().numpy().tobytes() == hp.alpha_rows_f64(reach, rto, rbar, GAMMA, V, act, vsel).tobytes()
    dev.close()


@pytest.mark.parametrize('O,R', [(2, 2), (5, 1)])
def test_plain_assemble_beyond_65535_tuples(torch_cuda, O, R):
    S, A, n = 6, 2, GRID_Y + 4465
    model = synthetic(S, A, O, R, seed=O * 10 + R)
    reach, _, rto, rbar = model
    rng = np.random.default_rng(O)
    V = 2.0 * rng.random((11, S)) - 1.0
    act = rng.integers(0, A, n).astype(np.int32)
    vsel = rng.integers(0, 11, (n, O)).astype(np.int32)
    dev = device(model)
    rows = dev.backup_assemble(V, GAMMA, act, vsel).cpu().numpy()
    assert launches(dev) == 1 + 2
    assert rows.tobytes() == hp.alpha_rows_f64(reach, rto, rbar, GAMMA, V, act, vsel).tobytes()
    dev.close()


# ---- Gamma projection in z-groups ------------------------------------------------------------------------------------------------
def test_gamma_projection_in_two_z_groups(torch_cuda):
    """R = 2, S = 20 000, nV = 2048, A = 4, O = 8: 32 (a, o) pairs of ~328 MB of Gamma each do not fit the 8 GB scratch at once, so the
    projection and the score kernel run in two groups (26 + 6) with shifted z orders; every z is checked."""
    S, A, O, R, nB, nV = 20000, 4, 8, 2, 16, 2048
    model = synthetic(S, A, O, R, seed=31)
    rng = np.random.default_rng(32)
    B = sparse_beliefs(rng, nB, S, [50, 17, 3, 1])
    V = rng.random((nV, S))
    Vp = -(-nV // 256) * 256
    z_group = max(1, min(A * O, (8 << 30) // ((S + 1) * Vp * 8)))
    groups = -(-(A * O) // z_group)
    assert groups == 2
    dev = device(model)
    rows, act, vstar, value = backup_checked(dev, model, B, V)
    vs2, val2, as2 = dev.backup_select(B, V, GAMMA)
    # transpose, alpha row mask, belief mask, chunk lists, (projection + score) per group, combine, approx, value pass, a*
    assert launches(dev) == 4 + 2 * groups + 4
    assert vs2.cpu().numpy().tobytes() == vstar.tobytes() and as2.cpu().numpy().tobytes() == act.tobytes()
    dev.close()


# ---- the small fused path --------------------------------------------------------------------------------------------------------
SMALL = [  # S, nV, A, O, R, nB
    (1, 1, 1, 3, 1, 8), (33, 31, 5, 2, 2, 40), (129, 32, 3, 3, 1, 30), (1024, 33, 1, 2, 1, 20), (129, 100, 6, 2, 2, 25),
    (33, 100, 2, 4, 1, 64), (1024, 1, 1, 3, 2, 12), (33, 33, 5, 1, 2, 50),
]


def small_checked(torch, dev, model, B, V):
    """backup_small == the exact decisions' rows (float64 restatement) after the ValueFunction dedup (first position, last action)."""
    reach, _, rto, rbar = model
    vstar, astar = exact_decisions(model, B, V)
    want = hp.alpha_rows_f64(reach, rto, rbar, GAMMA, V, astar, vstar[np.arange(len(B)), astar])
    want_rows, want_act, _ = orc.dedup_rows(want, astar)
    rows, acts, keys = dev.backup_small(torch.as_tensor(B, device='cuda'), torch.as_tensor(V, device='cuda'), GAMMA)
    assert rows.cpu().numpy().tobytes() == want_rows.tobytes()
    assert np.array_equal(acts, want_act)
    assert np.array_equal(keys, dev.row_hash(rows).cpu().numpy())


@pytest.mark.parametrize('S,nV,A,O,R,nB', SMALL)
def test_small_backup_against_the_reference(torch_cuda, S, nV, A, O, R, nB):
    """One block per belief, v over 32 lanes, z and a over 4 warps, s over 128 threads; R = 2 models land only on even states, so odd
    states have no predecessor in the landing-state CSR."""
    landing = np.arange(0, S, 2) if R > 1 else None
    model = synthetic(S, A, O, R, seed=S + nV + A, landing=landing)
    rng = np.random.default_rng(S * nV)
    B = sparse_beliefs(rng, nB, S, [S, 40, 5, 1])
    B[nB // 2] = B[0]                                         # repeated beliefs: repeated rows for the dedup
    V = rng.random((nV, S))
    dev = device(model)
    assert dev.backup_small_eligible(nB, nV) and dev._lib.pbvi_backup_small_eligible(dev._h, nB, nV) == 1
    small_checked(torch_cuda, dev, model, B, V)
    dev.close()


SMALL_BOUNDS = {  # bound: ((S, A, O, nB, nV) just inside, the same just outside)
    'S <= 1024': ((1024, 1, 2, 2, 2), (1025, 1, 2, 2, 2)),
    'shared memory (1 + A O) S + A + A O <= 5000': ((100, 4, 12, 2, 2), (101, 4, 12, 2, 2)),
    'nB S <= 262144': ((64, 1, 2, 4096, 2), (64, 1, 2, 4097, 2)),
    'nV <= 4096': ((4, 1, 2, 1, 4096), (4, 1, 2, 1, 4097)),
    'nB <= 16384': ((8, 1, 2, 16384, 3), (8, 1, 2, 16385, 3)),
    'nB nV A O S <= 6e7': ((100, 2, 2, 150, 1000), (100, 2, 2, 150, 1001)),
}


@pytest.mark.parametrize('bound', list(SMALL_BOUNDS))
def test_small_backup_eligibility_bounds(torch_cuda, bound):
    """Both sides of every bound of small_eligible: inside, the fused path runs and matches the reference; outside, the library
    refuses with PBVI_ERR_UNSUPPORTED (the host mirror agrees on both sides)."""
    from pomdp_pbvi_exploration_b200._native import PBVI_ERR_UNSUPPORTED
    torch = torch_cuda
    for inside, (S, A, O, nB, nV) in zip((True, False), SMALL_BOUNDS[bound]):
        model = synthetic(S, A, O, 1, seed=S + A * O)
        rng = np.random.default_rng(nB + nV)
        B = sparse_beliefs(rng, nB, S, [S, 5, 1])
        V = rng.random((nV, S))
        dev = device(model)
        assert dev.backup_small_eligible(nB, nV) == inside
        assert dev._lib.pbvi_backup_small_eligible(dev._h, nB, nV) == int(inside)
        if inside:
            small_checked(torch, dev, model, B, V)
        else:
            b, v = torch.as_tensor(B, device='cuda'), torch.as_tensor(V, device='cuda')
            out = torch.empty((nB, S), dtype=torch.float64, device='cuda')
            acts, keys, n = np.empty(nB, np.int32), np.empty((nB, 2), np.int64), ctypes.c_int(-1)
            rc = dev._lib.pbvi_backup_small(dev._h, b.data_ptr(), nB, v.data_ptr(), nV, GAMMA, out.data_ptr(), acts.ctypes.data,
                                            keys.ctypes.data, ctypes.byref(n), torch.cuda.current_stream().cuda_stream)
            assert rc == PBVI_ERR_UNSUPPORTED and n.value == 0
            assert b'too large' in dev._lib.pbvi_last_error()
        dev.close()


# ---- host chunking ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('nB', [2047, 2048, 2049, 4097])
def test_backup_host_chunks_equal_device_backup(torch_cuda, nB):
    """pbvi_backup_host walks the beliefs in chunks of 2048 rows: one row short of, exactly at, one row past a chunk, and a one-row
    third chunk; bytewise the rows and actions of pbvi_backup, which pass the contract."""
    model = synthetic(50, 3, 2, 1, seed=nB)
    rng = np.random.default_rng(nB)
    B = sparse_beliefs(rng, nB, 50, [50, 7, 1])
    V = rng.random((20, 50))
    dev = device(model)
    rows, act, _, _ = backup_checked(dev, model, B, V)
    hrows, hact = dev.backup_host(B, V, GAMMA)
    assert hrows.tobytes() == rows.tobytes() and hact.tobytes() == act.tobytes()
    dev.close()


# ---- GER -------------------------------------------------------------------------------------------------------------------------
def ger_checked(dev, B, succ, alpha_b, r_min, r_max):
    eps = dev.ger_scores(B, alpha_b, succ, r_min, r_max).cpu().numpy()
    ex, bd = hp.ger_eps(B, succ, alpha_b, r_min, r_max)
    nan = np.isnan(ex)
    assert nan.any()
    assert np.all(eps[nan] == 0.0)                            # an impossible observation contributes nothing
    hp.check_close(eps[~nan], ex[~nan], bd[~nan], what='GER eps')


@pytest.mark.parametrize('tag', ['hallway', 'olfactory_wrap'])
def test_ger_scores_against_the_reference(torch_cuda, tag):
    m, g = load_golden('model_' + tag), load_golden('backup_' + tag)
    reach = m['reach'].astype(np.int64)
    model = (reach, m['probs'] if 'probs' in m else None, m['rto'], m['rbar'])
    dev = device(model)
    B = g['beliefs'][:12]
    succ, _ = dev.belief_successors(B)
    succ = succ.cpu().numpy()
    succ[0, 0, 0] = np.nan                                    # at least one impossible observation
    _, best = orc.max_values(B, g['alphas'])
    gamma = float(m['gamma'])
    ger_checked(dev, B, succ, g['alphas'][best], -1.0 / (1 - gamma), 1.0 / (1 - gamma))
    dev.close()


def test_ger_scores_beyond_65535_beliefs(torch_cuda):
    m = load_golden('model_tiger')
    model = (m['reach'].astype(np.int64), m['probs'] if 'probs' in m else None, m['rto'], m['rbar'])
    dev = device(model)
    rng = np.random.default_rng(9)
    n = GRID_Y + 300
    B = rng.dirichlet(np.ones(2), size=n)
    succ, _ = dev.belief_successors(B)
    succ = succ.cpu().numpy()
    succ[n - 5, 1, 0] = np.nan
    alpha_b = 20.0 * rng.random((n, 2)) - 10.0
    ger_checked(dev, B, succ, alpha_b, -100.0, 10.0)
    dev.close()
