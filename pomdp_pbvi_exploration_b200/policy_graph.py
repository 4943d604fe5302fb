"""
Finite-state controllers (policy graphs) extracted from a value function, and their exact evaluation as a certified lower bound on V*.

    PolicyGraph   N nodes, node n playing action a_n and moving to node sigma(n, o) on observation o.  Its value vectors solve
                      V_n = Rbar_{a_n} + gamma * sum_o sum_r RTO[., a_n, o, r] * V_{sigma(n,o)}[reach[., a_n, r]]
                  and max_n V_n . b is the value of a policy that can be executed, hence a lower bound on V*(b) at every belief and for
                  every model, whatever the signs of its rewards.  `evaluate` iterates that fixed point on the device (one
                  persistent `pbvi_controller_evaluate` launch) and certifies the returned rows with a residual shift; `improve`
                  raises that bound by point-based policy iteration on the controller.  `outcomes` gives the exact success probability,
                  expected step count and return of runs that stop at end states, for every start (node, state) at once.

A graph may also have stochastic successor edges: a mixture is a convex combination of nodes, and a successor entry N + m means "move
to member k of mixture m with probability mu_k" (value-wise: the mixture row sum_k mu_k W_{node_k}).  `prune_lp` creates them when it
drops a node that a convex combination of other nodes dominates.

The file formats of `save` / `load` are pomdp-solve's: `.pg` ("id action succ_0 ... succ_{O-1}" per node) and `.alpha` (an action line, a
values line and a blank line per node), plus `.mix` ("mixture_id k node_1 weight_1 ... node_k weight_k" per mixture) for a graph with
mixtures.
"""
from __future__ import annotations

import os
import time

import numpy as np
import torch

from .bounds import belief_rows, certificate_contraction, resolve_witnesses
from .model import Model, log
from .solver import MDPSolverHistory
from .value_function import ValueFunction


def reachable_nodes(successors, roots, mixtures=None) -> np.ndarray:
    """bool [N]: the nodes a controller can reach from the nodes `roots`, through every edge (an impossible observation's included) and
    every member of a mixture that an edge names (successor entry N + m)."""
    succ = np.asarray(successors, dtype=np.int64)
    N = succ.shape[0]
    seen = np.zeros(N, dtype=bool)
    stack = sorted({int(r) for r in np.asarray(roots).reshape(-1)})
    seen[stack] = True
    while stack:
        for t in succ[stack.pop()].tolist():
            targets = [t] if t < N else mixtures[1][mixtures[0][t - N]:mixtures[0][t - N + 1]].tolist()
            for v in targets:
                if not seen[v]:
                    seen[v] = True
                    stack.append(v)
    return seen


def reachable_subgraph(actions, successors, roots) -> tuple:
    """
    The part of a controller that can run from the nodes `roots`: returns (kept node indices ascending, their actions, their successors
    renumbered to positions in the kept list).  Kept nodes keep their relative order, and every successor of a kept node is kept
    (whatever the observation, an impossible one included), so the rows of the kept nodes need no re-evaluation.
    """
    act = np.asarray(actions, dtype=np.int64).reshape(-1)
    succ = np.asarray(successors, dtype=np.int64)
    keep = np.flatnonzero(reachable_nodes(succ, roots))
    renumber = np.full(act.shape[0], -1, dtype=np.int64)
    renumber[keep] = np.arange(len(keep))
    return keep, act[keep], renumber[succ[keep]]


def redirect_dominated(actions, successors, witness) -> tuple:
    """
    Drops the nodes that have a witness (`pbvi_dominating_row`: a row >= theirs at every state) and sends every edge that pointed to a
    dropped node to the kept node at the end of its witness chain (`resolve_witnesses`), node-0 and impossible-observation edges
    included: returns (kept node indices ascending, their actions, their successors renumbered to positions in the kept list).
    """
    act = np.asarray(actions, dtype=np.int64).reshape(-1)
    succ = np.asarray(successors, dtype=np.int64)
    target = resolve_witnesses(witness)
    keep = np.flatnonzero(target == np.arange(act.shape[0]))
    renumber = np.full(act.shape[0], -1, dtype=np.int64)
    renumber[keep] = np.arange(len(keep))
    return keep, act[keep], renumber[target[succ[keep]]]


def check_mixtures(mixtures, N: int):
    """
    The validated mixture table of a graph with N nodes: (offsets int64 [M+1], nodes int64 [nnz], weights float64 [nnz]) with offsets
    rising strictly from 0 to nnz (no empty mixture), members in [0, N), finite weights >= 0 summing to 1 within 1e-12 per mixture.
    None, or a table with M = 0, gives None.  Raises ValueError otherwise.
    """
    if mixtures is None:
        return None
    if len(mixtures) != 3:
        raise ValueError('mixtures must be a tuple (offsets [M+1], nodes [nnz], weights [nnz])')
    off, nodes, w = (np.asarray(x).reshape(-1) for x in mixtures)
    if off.size == 0 or not np.issubdtype(off.dtype, np.integer) or (nodes.size and not np.issubdtype(nodes.dtype, np.integer)):
        raise ValueError('mixture offsets and nodes must be integer arrays, with at least one offset')
    off, nodes, w = off.astype(np.int64), nodes.astype(np.int64), w.astype(np.float64)
    if off.size == 1 and off[0] == 0 and nodes.size == 0 and w.size == 0:
        return None
    if off[0] != 0 or off[-1] != nodes.size or w.size != nodes.size or np.any(np.diff(off) <= 0):
        raise ValueError('mixture offsets must rise strictly from 0 to the number of members, with one weight per member')
    if nodes.min() < 0 or nodes.max() >= N:
        raise ValueError(f'mixture members must be nodes in [0, {N})')
    if not np.all(np.isfinite(w)) or w.min() < 0.0:
        raise ValueError('mixture weights must be finite and >= 0')
    sums = np.add.reduceat(w, off[:-1])
    if np.max(np.abs(sums - 1.0)) > 1e-12:
        raise ValueError('the weights of every mixture must sum to 1 (within 1e-12)')
    return off, nodes, w


def resolve_certificates(pruned, cert_idx, cert_w, drop: float = 1e-13, max_rounds: int = 100) -> dict:
    """
    The LP certificates of `pbvi_prune_lp_certificates` resolved onto kept nodes: pruned bool [n]; cert_idx [n, J] (-1 padded) and
    cert_w [n, J] the competitor sets and weights lambda of the pruned rows.  Returns {i: (nodes int64 ascending, weights float64)} for every
    pruned i whose resolution is non-empty: the weights on kept nodes of W_i's dominating combination, after substituting each pruned
    member j by its own combination (depth first, memoised; members that close a cycle are substituted again, in rounds, with the current
    resolutions).  Every certificate has a strict margin (its combination exceeds its row by more than tau everywhere), so no closed set of
    pruned rows keeps its weight among itself and the pruned mass decays geometrically.  What is left after `max_rounds`, and any weight
    below `drop`, is dropped and the rest renormalised: the result is a candidate, which `PolicyGraph.prune_lp` verifies on the device.
    """
    pruned = np.asarray(pruned, dtype=bool).reshape(-1)
    cert_idx, cert_w = np.asarray(cert_idx, dtype=np.int64), np.asarray(cert_w, dtype=np.float64)
    state = np.zeros(pruned.shape[0], dtype=np.int8)          # 0 new, 1 in progress, 2 resolved (possibly with cycle members left)
    res = {}

    def combine(nodes, weights):
        u, inv = np.unique(nodes, return_inverse=True)
        return u, np.bincount(inv, weights=weights, minlength=len(u))

    def substitute(nodes, weights, skip_in_progress):
        parts_n, parts_w = [nodes[~pruned[nodes]]], [weights[~pruned[nodes]]]
        for j, mu in zip(nodes[pruned[nodes]].tolist(), weights[pruned[nodes]].tolist()):
            if skip_in_progress and state[j] == 1:
                parts_n.append(np.asarray([j]))
                parts_w.append(np.asarray([mu]))
            else:
                rn, rw = res[j]
                parts_n.append(rn)
                parts_w.append(mu * rw)
        return combine(np.concatenate(parts_n), np.concatenate(parts_w))

    def visit(i):
        stack = [i]
        state[i] = 1
        while stack:
            top = stack[-1]
            sel = cert_idx[top] >= 0
            nxt = [j for j in cert_idx[top][sel].tolist() if pruned[j] and state[j] == 0]
            if nxt:
                state[nxt[0]] = 1
                stack.append(nxt[0])
                continue
            res[top] = substitute(cert_idx[top][sel], cert_w[top][sel], True)
            state[top] = 2
            stack.pop()

    for i in np.flatnonzero(pruned).tolist():
        if state[i] == 0:
            visit(i)
    for _ in range(max_rounds):
        left = [i for i, (nodes, weights) in res.items() if np.any(pruned[nodes])]
        if not left or all(float(np.sum(res[i][1][pruned[res[i][0]]])) <= drop for i in left):
            break
        for i in left:
            res[i] = substitute(*res[i], False)
    out = {}
    for i, (nodes, weights) in res.items():
        ok = ~pruned[nodes] & (weights > drop)
        if np.any(ok):
            out[i] = (nodes[ok], weights[ok] / np.sum(weights[ok]))
    return out


def mixture_rows(W: torch.Tensor, mixtures) -> torch.Tensor:
    """Z [M, S]: the mixture rows over node rows W in the arithmetic of the mixture phase of `pbvi_controller_evaluate_mixed`:
    z = mu_0 * W_0, then z = z + mu_k * W_k for the further members in stored order.  Each FP64 elementwise multiply and add rounds once
    (no FMA), as the kernel's __dmul_rn / __dadd_rn."""
    off, nodes, w = mixtures
    d = W.device
    lengths = np.diff(off)
    Z = torch.empty((len(lengths), W.shape[1]), dtype=torch.float64, device=d)
    for p in range(int(lengths.max()) if len(lengths) else 0):
        sel = np.flatnonzero(lengths > p)
        k = off[sel] + p
        t = W[torch.as_tensor(nodes[k], device=d)] * torch.as_tensor(w[k], dtype=torch.float64, device=d)[:, None]
        rows = torch.as_tensor(sel, device=d)
        Z[rows] = t if p == 0 else Z[rows] + t
    return Z


def compact_graph(actions, successors, redirect, mixtures=None, member_target=None) -> tuple:
    """
    A graph after dropping nodes.  redirect [N] sends the edges into each node to the node itself (it is kept), to another kept node, or
    to a mixture entry N + m of `mixtures` (which may hold more mixtures than the graph referenced so far); mixture members go to
    member_target [N] (default: redirect), which must name kept nodes.  Returns (kept node indices ascending, their actions, their
    successors, the mixtures that some kept edge references or None), nodes renumbered to positions in the kept list and the mixtures
    kept in their old order.
    """
    act = np.asarray(actions, dtype=np.int64).reshape(-1)
    succ = np.asarray(successors, dtype=np.int64)
    redirect = np.asarray(redirect, dtype=np.int64).reshape(-1)
    N = act.shape[0]
    keep = np.flatnonzero(redirect == np.arange(N))
    K = len(keep)
    renumber = np.full(N, -1, dtype=np.int64)
    renumber[keep] = np.arange(K)
    s = succ[keep]
    s = np.where(s < N, redirect[np.minimum(s, N - 1)], s)
    if mixtures is None:
        return keep, act[keep], renumber[s], None
    off, nodes, w = mixtures
    used = np.unique(s[s >= N]) - N
    mix_renumber = np.full(len(off) - 1, -1, dtype=np.int64)
    mix_renumber[used] = np.arange(len(used))
    target = redirect if member_target is None else np.asarray(member_target, dtype=np.int64).reshape(-1)
    sel = np.concatenate([np.arange(off[m], off[m + 1]) for m in used]) if len(used) else np.zeros(0, dtype=np.int64)
    out = np.where(s < N, renumber[np.minimum(s, N - 1)], K + mix_renumber[np.maximum(s - N, 0)])
    if not len(used):
        return keep, act[keep], out, None
    table = (np.concatenate([[0], np.cumsum(np.diff(off)[used])]), renumber[target[nodes[sel]]], w[sel])
    return keep, act[keep], out, table


def backup_tuples(dev, beliefs: torch.Tensor, rows: torch.Tensor, gamma: float) -> np.ndarray:
    """The backup tuple t_b = (a*_b, v*[b, a*_b, 0..O-1]) of every belief against the node rows (`backup_select`): int64 [nB, 1 + O].
    Read as a controller node, t_b plays a*_b and moves to node v*[b, a*_b, o] on o (an impossible observation scores zero everywhere,
    so it leads to node 0)."""
    vstar, _, astar = dev.backup_select(beliefs, rows, gamma, want_value=False)
    idx = torch.arange(beliefs.shape[0], device=astar.device)
    return torch.cat([astar[:, None], vstar[idx, astar.long()]], dim=1).cpu().numpy().astype(np.int64)


def node_index(actions, successors) -> dict:
    """(action, successor_0, ..., successor_{O-1}) -> node, the first node with a given tuple winning."""
    node_of = {}
    for n in range(len(actions) - 1, -1, -1):
        node_of[(int(actions[n]), *successors[n].tolist())] = n
    return node_of


def match_tuples(node_of: dict, tuples: np.ndarray) -> tuple:
    """Splits backup tuples [n, 1 + O] into the nodes that already play one (a set) and the distinct other tuples in order of first
    occurrence (int64 [m, 1 + O])."""
    in_use, new = set(), {}
    for t in map(tuple, tuples.tolist()):
        if t in node_of:
            in_use.add(node_of[t])
        elif t not in new:
            new[t] = len(new)
    return in_use, np.asarray(list(new), dtype=np.int64).reshape(-1, tuples.shape[1])


BPI_COLUMNS = 64                   # columns of one restricted master LP (J_MAX of pbvi_bpi_lp)
BPI_POOL_BYTES = 2 << 30           # worst-case column pool of one batch of nodes
BPI_POOL_ROWS = BPI_COLUMNS + 2    # per node: its row, its own row, 63 appended columns and the last one priced (checked, not appended)
BPI_DROP = 1e-13                   # LP weights below this are dropped before the graph surgery


def bpi_lps(dev, W: torch.Tensor, own: torch.Tensor, gamma: float, tau: float, batch: int | None = None) -> dict:
    """
    The restricted master LPs of bounded policy iteration for every node, by column generation: node n's LP is
    max eps s.t. sum_t lambda_t Y_t >= W_n + eps, sum lambda = 1, lambda >= 0 over the columns generated so far, started from its own
    one-sweep row own[n].  Each round runs `pbvi_bpi_lp` on the batch, then prices every still active node with one `backup_select` at its
    tangent belief b* (the best tuple t* = argmax_t b* . Y_t), assembles the tuples that are new to the batch (`backup_assemble`, one row
    per distinct tuple) into the pool and hands each node its t*.  Nodes go in batches of `batch` (default: the pool of a batch stays under
    BPI_POOL_BYTES); an entry's results depend on its own rows and columns only, so they are bitwise the same for every batch split.

    Returns status int64 [N] (1 not improvable, 2 optimal, 3 budget, 4 numerical), delta / u / mstar float64 [N] (delta_J of the last LP,
    its verified bound max_s (W_n - sum lambda Y)[s], b* . (W_n - Y_{t*}) of the last check), lam float64 [N, 64], columns int64 [N, 64]
    (-1 the node's own row, t >= 0 row t of `tuples`, -2 padding), tuples int64 [T, 1 + O] (action, successor nodes), bstar CUDA float64
    [N, S], stats {rounds, max_columns, lps, pivots, pool_rows} and seconds {lp, select, assemble}.
    """
    N, S = W.shape
    d = W.device
    if batch is None:
        batch = max(1, BPI_POOL_BYTES // (BPI_POOL_ROWS * S * 8))
    out = dict(status=np.zeros(N, np.int64), delta=np.zeros(N), u=np.zeros(N), mstar=np.zeros(N), lam=np.zeros((N, BPI_COLUMNS)),
               columns=np.full((N, BPI_COLUMNS), -2, np.int64), bstar=torch.zeros((N, S), dtype=torch.float64, device=d))
    tuple_id = {}
    stats = dict(rounds=0, max_columns=0, lps=0, pivots=0, pool_rows=0)
    sec = dict(lp=0.0, select=0.0, assemble=0.0)
    for lo in range(0, N, batch):
        hi = min(N, lo + batch)
        n = hi - lo
        pool = torch.empty((BPI_POOL_ROWS * n, S), dtype=torch.float64, device=d)
        pool[:n], pool[n:2 * n] = W[lo:hi], own[lo:hi]
        P = 2 * n
        row_tuple = {}                                     # tuple -> pool row
        tuples_of_row = {}                                 # pool row -> tuple
        i32 = dict(dtype=torch.int32, device=d)
        f64 = dict(dtype=torch.float64, device=d)
        corner = torch.argmax(W[lo:hi] - own[lo:hi], dim=1).to(torch.int32).contiguous()
        price = torch.full((n,), -1, **i32)
        cols = torch.full((n, BPI_COLUMNS), -1, **i32)
        cols[:, 0] = torch.arange(n, 2 * n, **i32)
        ncols = torch.ones((n,), **i32)
        bstar = torch.zeros((n, S), **f64)
        delta, u, mstar = (torch.full((n,), float('nan'), **f64) for _ in range(3))
        lam = torch.zeros((n, BPI_COLUMNS), **f64)
        status = torch.full((n,), -1, **i32)
        while True:
            t0 = time.perf_counter()
            st = dev.bpi_lp(pool, n, tau, corner, price, cols, ncols, bstar, delta, u, lam, mstar, status)
            sec['lp'] += time.perf_counter() - t0
            stats['rounds'] += 1
            stats['max_columns'] = max(stats['max_columns'], st['max_columns'])
            stats['lps'] += st['lps']
            stats['pivots'] += st['pivots']
            active = np.flatnonzero(status.cpu().numpy() == -1)
            if not len(active):
                break
            t0 = time.perf_counter()
            tup = backup_tuples(dev, bstar[torch.as_tensor(active, device=d)], W, gamma)
            sec['select'] += time.perf_counter() - t0
            t0 = time.perf_counter()
            rows, new = np.empty(len(active), np.int64), []
            for k, t in enumerate(map(tuple, tup.tolist())):
                if t not in row_tuple:
                    row_tuple[t] = P + len(new)
                    tuples_of_row[P + len(new)] = t
                    new.append(t)
                rows[k] = row_tuple[t]
            if new:
                assert P + len(new) <= pool.shape[0]           # every active node adds at most one column per round
                nt = np.asarray(new, dtype=np.int64)
                pool[P:P + len(new)] = dev.backup_assemble(W, gamma, nt[:, 0], nt[:, 1:])
                P += len(new)
            price[torch.as_tensor(active, device=d)] = torch.as_tensor(rows, **i32)
            torch.cuda.synchronize(d)
            sec['assemble'] += time.perf_counter() - t0
        stats['pool_rows'] = max(stats['pool_rows'], P)
        k = ncols.cpu().numpy()
        c = cols.cpu().numpy()
        for j in range(n):
            for q in range(int(k[j])):
                r = int(c[j, q])
                if q == 0:
                    out['columns'][lo + j, q] = -1
                else:
                    t = tuples_of_row[r]
                    out['columns'][lo + j, q] = tuple_id.setdefault(t, len(tuple_id))
        out['status'][lo:hi] = status.cpu().numpy()
        out['delta'][lo:hi], out['u'][lo:hi], out['mstar'][lo:hi] = delta.cpu().numpy(), u.cpu().numpy(), mstar.cpu().numpy()
        out['lam'][lo:hi] = lam.cpu().numpy()
        out['bstar'][lo:hi] = bstar
    out['tuples'] = np.asarray(list(tuple_id), dtype=np.int64).reshape(len(tuple_id), -1) if tuple_id else None
    out['stats'], out['seconds'] = stats, sec
    return out


def successor_distribution(entry: int, N: int, mixtures) -> tuple:
    """(members, weights) of a successor entry: node t is ([t], [1]), mixture entry N + m its members (a flattened mixture)."""
    if entry < N:
        return np.asarray([entry], np.int64), np.ones(1)
    off, nodes, w = mixtures
    m = entry - N
    return nodes[off[m]:off[m + 1]], w[off[m]:off[m + 1]]


def combine_members(nodes, weights) -> tuple:
    """Duplicate members merged (ascending) and the weights renormalised to sum 1."""
    u, inv = np.unique(np.asarray(nodes, np.int64), return_inverse=True)
    w = np.bincount(inv, weights=np.asarray(weights, np.float64), minlength=len(u))
    return u, w / w.sum()


def bpi_split(columns, lam, N: int, mixtures, drop: float = BPI_DROP) -> list:
    """
    The nodes that replace an improved node: `columns` = [(action, successor entries [O])] of its LP solution, `lam` their weights.
    Weights below `drop` are dropped and the rest renormalised; per action a (ascending) the node n_a plays a and on o moves to the
    distribution {sigma_t(o) : a_t = a} with weights lambda_t / c_a (mixture entries flattened into their members, duplicates merged).
    Returns [(a, c_a, [(members, weights) per o])], the c_a summing to 1.
    """
    lam = np.asarray(lam, np.float64)
    keep = np.flatnonzero(lam >= drop)
    lam = lam[keep] / lam[keep].sum()
    cols = [columns[k] for k in keep]
    acts = np.asarray([a for a, _ in cols], np.int64)
    out = []
    for a in np.unique(acts).tolist():
        idx = np.flatnonzero(acts == a)
        c = float(lam[idx].sum())
        O = len(cols[idx[0]][1])
        edges = []
        for o in range(O):
            parts = [successor_distribution(int(cols[k][1][o]), N, mixtures) for k in idx]
            edges.append(combine_members(np.concatenate([p[0] for p in parts]),
                                         np.concatenate([p[1] * (lam[k] / c) for p, k in zip(parts, idx)])))
        out.append((a, c, edges))
    return out


def bpi_assemble(actions, successors, mixtures, splits: dict, redirect: bool) -> tuple:
    """
    A graph with the nodes of `splits` ({n: bpi_split(...)}) added.  redirect=False (the graph the start rows are swept on): every
    split node is appended and no old edge changes.  redirect=True (the improved graph): n_{a_0} of the first action takes n's index and
    the others are appended, and every edge or mixture member naming a split node n with more than one action goes to the mixture
    {n_a : c_a} instead (members flattened).  Old mixtures keep their ids (members rewritten when they name such an n); further mixtures
    are appended, one per distinct distribution.  Returns (actions, successors, mixtures or None, {(n, j): node index of n's j-th split}).
    """
    act = np.asarray(actions, np.int64)
    succ = np.asarray(successors, np.int64)
    N, O = succ.shape
    pos, extra = {}, N
    for n in sorted(splits):
        for j in range(len(splits[n])):
            if redirect and j == 0:
                pos[(n, 0)] = n
            else:
                pos[(n, j)] = extra
                extra += 1
    N2 = extra
    sub = {n: (np.asarray([pos[(n, j)] for j in range(len(sp))]), np.asarray([c for _, c, _ in sp]))
           for n, sp in splits.items() if redirect and len(sp) > 1}

    def substitute(nodes, weights):
        if not any(int(t) in sub for t in nodes):
            return nodes, weights
        parts = [sub[int(t)] if int(t) in sub else (np.asarray([t]), np.ones(1)) for t in nodes]
        return combine_members(np.concatenate([p[0] for p in parts]), np.concatenate([p[1] * w for p, w in zip(parts, weights)]))

    table, index = [], {}
    M = 0 if mixtures is None else len(mixtures[0]) - 1
    for m in range(M):
        table.append(substitute(*successor_distribution(N + m, N, mixtures)))

    def intern(nodes, weights):
        key = (tuple(nodes.tolist()), tuple(weights.tolist()))
        if key not in index:
            index[key] = len(table)
            table.append((nodes, weights))
        return index[key]

    target = np.arange(N)
    for n in sorted(sub):
        target[n] = N2 + intern(*sub[n])
    act2 = np.concatenate([act, np.zeros(N2 - N, np.int64)])
    succ2 = np.zeros((N2, O), np.int64)
    succ2[:N] = np.where(succ < N, target[np.minimum(succ, N - 1)], N2 + succ - N)
    for n in sorted(splits):
        for j, (a, _, edges) in enumerate(splits[n]):
            k = pos[(n, j)]
            act2[k] = a
            for o, (nodes, weights) in enumerate(edges):
                nodes, weights = substitute(nodes, weights)
                succ2[k, o] = int(nodes[0]) if len(nodes) == 1 else N2 + intern(nodes, weights)
    if not table:
        return act2, succ2, None, pos
    off = np.concatenate([[0], np.cumsum([len(t[0]) for t in table])]).astype(np.int64)
    mix = (off, np.concatenate([t[0] for t in table]).astype(np.int64), np.concatenate([t[1] for t in table]).astype(np.float64))
    return act2, succ2, mix, pos


NO_MIXTURES = (np.zeros(1, np.int64), np.zeros(0, np.int64), np.zeros(0))


class ControllerOutcomes:
    """
    What `PolicyGraph.outcomes` returns for q query pairs (belief b_j, start node n_j) and horizon H:
        start_nodes                                    int64 [q]
        success, steps, discounted_return              float64 [q]: P(T <= H), E[min(T, H)] and E[sum_{t < min(T, H)} gamma^t r_t] at b_j
        success_curve, steps_curve, return_curve       float64 [q, H] (NumPy): the same after k = 1..H steps (column k - 1)
        success_rows, steps_rows, return_rows          CUDA float64 [N, S]: the values at H of a run started in (node, true state)
    """

    def __init__(self, start_nodes, series: np.ndarray, rows: tuple, gamma: float, max_steps: int):
        self.start_nodes = np.asarray(start_nodes, dtype=np.int64)
        self.gamma, self.max_steps = gamma, max_steps
        curves = np.ascontiguousarray(np.transpose(series, (1, 2, 0)))                       # [q, 3, H]
        self.success_curve, self.steps_curve, self.return_curve = curves[:, 0], curves[:, 1], curves[:, 2]
        last = curves[:, :, -1] if max_steps > 0 else np.zeros((len(self.start_nodes), 3))
        self.success, self.steps, self.discounted_return = last[:, 0].copy(), last[:, 1].copy(), last[:, 2].copy()
        self.success_rows, self.steps_rows, self.return_rows = rows


class PolicyGraph:
    """
    A finite-state controller over `model`: `actions` [N] and `successors` [N, O] (node indices) as host int64 arrays; after `evaluate` (or
    `load` of a saved graph with rows) `rows` [N, S] is a CUDA float64 tensor of node values.  `source_rows` [N] holds, for an extracted
    graph, the row of the value function each node came from (None otherwise).

    `mixtures` (optional): stochastic successor edges as a CSR table (offsets [M+1], nodes [nnz], weights [nnz]) -- mixture m moves to
    node nodes[k] with probability weights[k] for k in [offsets[m], offsets[m+1]) (members in [0, N), FP64 weights >= 0 summing to 1
    within 1e-12) -- and a successor entry N + m means "mixture m".  Stored as host int64 / int64 / float64 arrays, or None.
    """

    def __init__(self, model: Model, actions, successors, rows=None, source_rows=None, mixtures=None):
        self.model = model
        A, O, S = model.action_count, model.observation_count, model.state_count
        act = np.asarray(actions).astype(np.int64).reshape(-1)
        succ = np.asarray(successors).astype(np.int64)
        N = act.shape[0]
        if N < 1:
            raise ValueError('a policy graph needs at least one node')
        if succ.shape != (N, O):
            raise ValueError(f'successors must be [{N}, {O}], got {tuple(succ.shape)}')
        if act.min() < 0 or act.max() >= A:
            raise ValueError(f'node actions must lie in [0, {A})')
        self.mixtures = check_mixtures(mixtures, N)
        M = 0 if self.mixtures is None else len(self.mixtures[0]) - 1
        if succ.min() < 0 or succ.max() >= N + M:
            raise ValueError(f'successor entries must lie in [0, {N + M}) ({N} nodes, {M} mixtures)')
        self.actions, self.successors = act, succ
        self.source_rows = None if source_rows is None else np.asarray(source_rows).astype(np.int64).reshape(-1)
        self.rows = None
        if rows is not None:
            self.rows = torch.as_tensor(np.asarray(rows, dtype=np.float64) if not isinstance(rows, torch.Tensor) else rows)
            self.rows = self.rows.to(device=model.device.device, dtype=torch.float64).contiguous()
            if tuple(self.rows.shape) != (N, S):
                raise ValueError(f'rows must be [{N}, {S}], got {tuple(self.rows.shape)}')
        self._initial = None           # [N, S] start of `evaluate` (the source rows of an extracted graph)
        self.witnesses = None          # [N, S] of an extracted graph: the belief at which each node's row was chosen
        self._value_function = None
        self.gamma = None              # discount of the last `evaluate`
        self.prune_stats = None        # of a graph that `prune_lp` returned

    def __len__(self) -> int:
        return int(self.actions.shape[0])

    # ---- construction -----------------------------------------------------------------------------------------------------
    @classmethod
    def blind(cls, model: Model) -> 'PolicyGraph':
        """A nodes, node a playing action a forever: the blind-policy lower bound."""
        A, O = model.action_count, model.observation_count
        return cls(model, np.arange(A), np.repeat(np.arange(A)[:, None], O, axis=1))

    @classmethod
    def from_value_function(cls, model: Model, value_function: ValueFunction, beliefs=None) -> tuple:
        """
        The controller that follows `value_function`: returns (PolicyGraph, stats dict with `nodes`, `closure_rounds`, `seconds`).

        A node is a row of the value function, playing that row's action; it is created at a witness belief where the row is the
        (first) argmax.  The start witnesses are b0 and then the rows of `beliefs`: the best row at each becomes a node, in order of first
        occurrence.  sigma(n, o) is the node of v*[w_n, a_n, o], the best row at the successor of w_n under (a_n, o) (one
        `backup_select` over the witnesses of the nodes added in a round); a row that is not a node yet becomes one, with the normalised
        successor belief as its witness (nodes in node order, o ascending: the first witness found wins).  Repeated until closed, at most
        |V| rounds.  An observation that is impossible at w_n leads to node 0.  Any successor choice gives a valid controller: these
        rules decide the quality of the bound, never its soundness.
        """
        t0 = time.perf_counter()
        dev = model.device
        rows = value_function.alpha_vector_array.contiguous()
        labels = np.asarray(value_function.actions, dtype=np.int64)
        if rows.shape[0] == 0 or not bool(torch.isfinite(rows).all()):
            raise ValueError('the value function must have at least one row and finite entries')
        W0 = belief_rows(model, model.start_probabilities)
        if beliefs is not None:
            W0 = torch.cat([W0, belief_rows(model, beliefs)])
        best = dev.max_values(W0, rows)[1].cpu().numpy()
        node_of = {}                   # value-function row -> node
        src, wit = [], []
        for j, v in enumerate(best.tolist()):
            if v not in node_of:
                node_of[v] = len(src)
                src.append(v)
                wit.append(j)
        witnesses = [W0[torch.as_tensor(wit, device=W0.device)]]
        O = model.observation_count
        succ_rows = []                 # per round: [p, O] successor nodes of the nodes added in the round before
        lo, rounds = 0, 0
        while lo < len(src):
            rounds += 1
            hi = len(src)
            Wp = witnesses[-1]
            acts = labels[src[lo:hi]]
            idx = torch.arange(hi - lo, device=Wp.device)
            a_t = torch.as_tensor(acts, device=Wp.device)
            # v* is the argmax of b^{ao} . alpha over the rows; gamma only scales the scores, so any positive value gives the same v*
            vstar = dev.backup_select(Wp, rows, 1.0, want_value=False)[0][idx, a_t].cpu().numpy()
            mass = dev.observation_probabilities(Wp)[idx, a_t].cpu().numpy()
            out = np.zeros((hi - lo, O), dtype=np.int64)
            new_k, new_o = [], []
            for k in range(hi - lo):
                for o in range(O):
                    if not mass[k, o] > 0.0:
                        continue                                   # impossible observation: node 0
                    v = int(vstar[k, o])
                    node = node_of.get(v)
                    if node is None:
                        node = node_of[v] = len(src)
                        src.append(v)
                        new_k.append(k)
                        new_o.append(o)
                    out[k, o] = node
            succ_rows.append(out)
            if new_k:
                b, _ = dev.belief_update(Wp[torch.as_tensor(new_k, device=Wp.device)], acts[new_k], np.asarray(new_o), normalise=True)
                witnesses.append(b)
            lo = hi
        src_np = np.asarray(src, dtype=np.int64)
        pg = cls(model, labels[src_np], np.concatenate(succ_rows), source_rows=src_np)
        pg._initial = rows[torch.as_tensor(src_np, device=rows.device)].contiguous()
        pg.witnesses = torch.cat(witnesses)
        stats = dict(nodes=len(pg), closure_rounds=rounds, seconds=time.perf_counter() - t0)
        return pg, stats

    # ---- evaluation -------------------------------------------------------------------------------------------------------
    def evaluate(self, gamma: float, eps: float = 1e-6, max_sweeps: int = 100000, print_progress: bool = False) -> tuple:
        """
        Certified node values: returns (rows [N, S] CUDA float64, MDPSolverHistory with `sweeps`, `final_change`, `residual`, `shift`).

        Iterates W <- T_pi W (`pbvi_controller_evaluate`: every sweep in one persistent launch, synchronised once) from the source rows
        (the Rbar rows of the node actions for a graph without them; the start `improve` sets) until max |T_pi W - W| <
        eps * gamma / (1 - gamma) or `max_sweeps` sweeps.  A graph with mixtures runs `pbvi_controller_evaluate_mixed`, whose sweeps
        read a mixture successor as the mixture row sum_k mu_k W_{node_k}; the certificate is the same.  Certificate, the
        mirror image of FIB_Solver's: with e = max(W - T_pi W) and gamma' = gamma * max(1, max_{s,a} sum_{o,r} RTO) the returned rows are
        W - max(e, 0) / (1 - gamma').  A constant shift c >= 0 passes through T_pi as at most gamma' * c, so they satisfy W <= T_pi W; they
        are re-checked with one more sweep, and while rounding leaves a positive residual e' the rows are lowered again by
        (e' + a few ulps of max |W|) / (1 - gamma') (three rounds at most, then ValueError).  T_pi is monotone and a gamma'-contraction, so every returned row lies below the value of the controller
        started in its node: max_n W_n . b <= V*(b).  gamma' >= 1 raises ValueError.
        """
        gamma = float(gamma)
        if not 0.0 < gamma < 1.0:
            raise ValueError('gamma must lie in (0, 1)')
        gamma_c = certificate_contraction(self.model, gamma, 'controller')
        dev = self.model.device
        d = dev.device
        act = torch.as_tensor(self.actions, dtype=torch.int32, device=d)
        succ = torch.as_tensor(self.successors, dtype=torch.int32, device=d).contiguous()
        if self._initial is not None:
            W = self._initial
        else:
            rbar = torch.as_tensor(np.asarray(self.model.expected_rewards_table, dtype=np.float64), device=d)
            W = rbar.T[act.long()].contiguous()
        history = MDPSolverHistory(1, self.model, gamma, eps, None)
        tol = eps * gamma / (1.0 - gamma)
        change = float('nan')
        if max_sweeps >= 1:
            # the whole iteration is one persistent launch; the sweeps are not timed one by one, so each gets an even share of the wall time
            start = time.perf_counter()
            if self.mixtures is None:
                W, changes, k = dev.controller_evaluate(W, gamma, act, succ, tol, max_sweeps)
            else:
                W, changes, k = dev.controller_evaluate_mixed(W, gamma, act, succ, self.mixtures, tol, max_sweeps)
            changes = changes.cpu().numpy().tolist()
            per_sweep = (time.perf_counter() - start) / k
            for c in changes:
                history.add(per_sweep, c, None)
            change = changes[-1]
            if change != change:
                raise ValueError('the controller iterates are not finite')
        residual = self._residual(W, gamma, act, succ)
        if residual != residual:
            raise ValueError('the controller iterates are not finite')
        shift = max(residual, 0.0) / (1.0 - gamma_c)
        if shift > 0.0:
            W = W - shift
        # what is left after the shift is rounding: it is taken off together with a rounding allowance of (O*R + 2) ulps of the largest
        # entry, so that the next check is not left to the same coin flip
        m = self.model
        ulps = (m.observation_count * m.reachable_state_count + 2) * 2.0 ** -52
        for _ in range(3):
            left = self._residual(W, gamma, act, succ)
            if not left > 0.0:
                break
            extra = (left + ulps * float(torch.max(torch.abs(W)))) / (1.0 - gamma_c)
            W = W - extra
            shift += extra
        else:
            raise ValueError(f'the controller certificate did not close: max(W - T W) = {left:.3e} after three shifts')
        history.sweeps, history.final_change, history.residual, history.shift = len(history.iteration_times), change, residual, shift
        self.rows, self.gamma, self._value_function = W.contiguous(), gamma, None
        if print_progress:
            log(f'PolicyGraph: {len(self)} nodes, {history.sweeps} sweeps, residual max(W - TW) = {residual:.3e}, certificate shift {shift:.3e}')
        return self.rows, history

    def _residual(self, W, gamma, act, succ) -> float:
        """max(W - T_pi W) over every entry (NaN wins) from one sweep: `pbvi_controller_sweep`'s stats, or for a graph with mixtures one
        sweep of `pbvi_controller_evaluate_mixed` (W - out rounds as -(out - W), so it is the same quantity)."""
        dev = self.model.device
        if self.mixtures is None:
            return float(dev.controller_sweep(W, gamma, act, succ, want_stats=True)[1][1])
        out = dev.controller_evaluate_mixed(W, gamma, act, succ, self.mixtures, float('inf'), 1)[0]
        d = W - out
        return float('nan') if bool(torch.isnan(d).any()) else float(d.max())

    # ---- improvement -------------------------------------------------------------------------------------------------------
    def improve(self, beliefs, iterations: int = 1, eps: float = 1e-6) -> tuple:
        """
        Point-based policy iteration (Hansen 1998; Ji et al. 2007) over B = b0 followed by the rows of `beliefs`: returns (PolicyGraph,
        list of per-iteration stats dicts).  Needs an evaluated graph (`rows`, `gamma`).  Each iteration, with W the certified node rows:

          1. backup: `backup_select(B, W)` gives at each b the tuple t_b = (a*_b, v*[b, a*_b, :]), a controller node that plays a*_b and
             moves to node v*[b, a*_b, o] on o (an impossible observation scores zero everywhere, so it leads to node 0).  Distinct tuples
             in order of first occurrence; a tuple equal to a node's (action, successors) is that node (the first such).
          2. rows: Y = `backup_assemble(W)` of the tuples that are not nodes yet.
          3. Hansen's rule (`first_dominating_row(Y, W)`): an old node dominated by some Y_j takes tuple j's action and successors and keeps
             its index -- unless some t_b is that node, which stays as it is; a tuple that dominated no node is appended.  The start of the
             next evaluation is X = W on the old nodes and Y_j on the appended ones.
          4. `evaluate(gamma, eps)` from X, with its certificate.
          5. prune: only the nodes reachable from the argmax nodes at B (`max_values` on the certified rows) are kept, renumbered in their
             old order (`reachable_subgraph`).  Kept nodes point to kept nodes only, so their rows are a subset and stay certified.
        An iteration that appends and overwrites nothing is the policy-iteration fixed point at B: the graph comes back unchanged.

        Why the bound rises: successors always name old nodes, and X equals W on every old node.  So (T_new X)_n is (T_old W)_n >= W_n
        (the certificate) for an untouched node, Y_j >= W_n for an overwritten one and Y_j = X_n for an appended one: X <= T_new X.  T_new
        is monotone and a contraction, so the new controller's value V satisfies V >= T_new X >= X.  Every t_b is played by some node m
        with (T_new X)_m = Y_{t_b}, so at every b in B the new value is >= the backup value Y_{t_b} . b >= (T_old W)_n . b >= W_n . b for
        the old argmax node n at b: the old value.  All of this holds in exact arithmetic; the certified rows of step 4 can lie below V
        by their shift, and that is what a caller sees at most as a fall.  Pruning keeps the argmax nodes of B and everything they reach.

        Stats per iteration: nodes_before, nodes_after, appended, overwritten, pruned, sweeps, value_b0 (certified), shift and
        seconds {select, assemble, dominance, evaluate, prune}.  A graph with mixtures raises ValueError.
        """
        self._require_rows()
        if self.gamma is None:
            raise ValueError('improve needs the gamma of evaluate: call evaluate(gamma) first')
        if self.mixtures is not None:
            raise ValueError('improve needs a graph without mixtures: it keys nodes by deterministic (action, successors) tuples')
        m, gamma = self.model, self.gamma
        dev = m.device
        B = belief_rows(m, m.start_probabilities)
        if beliefs is not None:
            B = torch.cat([B, belief_rows(m, beliefs)])
        pg, all_stats = self, []
        for _ in range(int(iterations)):
            W, N = pg.rows, len(pg)
            sec = {}
            t0 = time.perf_counter()
            tuples = backup_tuples(dev, B, W, gamma)
            sec['select'] = time.perf_counter() - t0
            t0 = time.perf_counter()
            node_of = node_index(pg.actions, pg.successors)
            in_use, new_t = match_tuples(node_of, tuples)
            Y = dev.backup_assemble(W, gamma, new_t[:, 0], new_t[:, 1:]) if len(new_t) else None
            torch.cuda.synchronize(dev.device)
            sec['assemble'] = time.perf_counter() - t0
            t0 = time.perf_counter()
            dom = dev.first_dominating_row(Y, W).cpu().numpy() if Y is not None else np.full(N, -1)
            sec['dominance'] = time.perf_counter() - t0
            actions, successors = pg.actions.copy(), pg.successors.copy()
            used = np.zeros(len(new_t), dtype=bool)
            overwritten = 0
            for n in range(N):
                j = int(dom[n])
                if j >= 0 and n not in in_use:
                    actions[n], successors[n] = new_t[j, 0], new_t[j, 1:]
                    used[j] = True
                    overwritten += 1
            app = np.flatnonzero(~used)
            stats = dict(nodes_before=N, appended=int(len(app)), overwritten=overwritten)
            if len(app) == 0 and overwritten == 0:
                stats.update(nodes_after=N, pruned=0, sweeps=0, value_b0=float(pg.value(B[:1])[0][0]), shift=0.0,
                             seconds=dict(sec, evaluate=0.0, prune=0.0))
                all_stats.append(stats)
                break
            t0 = time.perf_counter()
            nxt = PolicyGraph(m, np.concatenate([actions, new_t[app, 0]]), np.concatenate([successors, new_t[app, 1:]]))
            nxt._initial = torch.cat([W, Y[torch.as_tensor(app, device=W.device)]]).contiguous() if len(app) else W
            rows, hist = nxt.evaluate(gamma, eps)
            sec['evaluate'] = time.perf_counter() - t0
            t0 = time.perf_counter()
            roots = dev.max_values(B, rows)[1].cpu().numpy()
            keep, k_act, k_succ = reachable_subgraph(nxt.actions, nxt.successors, roots)
            pg = PolicyGraph(m, k_act, k_succ, rows=rows[torch.as_tensor(keep, device=rows.device)])
            pg.gamma = gamma
            sec['prune'] = time.perf_counter() - t0
            stats.update(nodes_after=len(pg), pruned=len(nxt) - len(pg), sweeps=hist.sweeps, value_b0=float(pg.value(B[:1])[0][0]),
                         shift=hist.shift, seconds=sec)
            all_stats.append(stats)
        return pg, all_stats

    def bounded_improve(self, beliefs=None, iterations: int = 1, eps: float = 1e-6) -> tuple:
        """
        Bounded policy iteration (Poupart & Boutilier 2003) on the controller: returns (PolicyGraph, list of per-iteration stats dicts).
        Needs an evaluated graph (`rows`, `gamma`); graphs with mixtures are accepted.  Each iteration, with W the certified node rows
        (W <= T_pi W) and a tuple t = (a, sigma(0..O-1)) a node that plays a and moves to node sigma(o), with row Y_t = backup_assemble(W, t):

          1. LP: for every node n, max eps s.t. sum_t lambda_t Y_t[s] >= W_n[s] + eps at every s, sum lambda = 1, lambda >= 0, over all
             A * N^O tuples.  In belief space this is delta = max_{b in simplex} min_t b . (W_n - Y_t), eps = -delta: the restricted LP
             of `pbvi_prune_lp` with columns Y_t as competitors, generated by `bpi_lps`.  J starts with n's own one-sweep row
             (T_pi W)_n >= W_n (for a node with mixture edges the mixed sweep's row, not a deterministic tuple) and the seed corner
             argmax_s (W_n - Y_own)[s].  Pricing: at the LP's tangent belief b* the best column over all tuples is the point-based backup
             at b* (one `backup_select` row), and m* = b* . (W_n - Y_t*) <= delta <= delta_J.  The search stops when m* > -tau (n cannot
             be improved by more than tau; b* is its tangent belief), when m* >= delta_J - tau (the LP is optimal), or at 64 columns or
             the pivot budget (the last LP stands).  n is improved when the last LP's verified bound u = max_s (W_n - sum lambda Y_J)[s]
             is < -tau, with tau = 1e-9 * max(1, max |W|, max |T_pi W|).
          2. Surgery (`bpi_split`, `bpi_assemble`): weights below 1e-13 are dropped; per action a of the solution, c_a = the weight of
             its columns and n_a plays a and on o moves to the mixture {sigma_t(o) : a_t = a} with weights lambda_t / c_a (the own
             column contributes n's own successor entries, mixtures flattened).  X_{n_a} = one mixed sweep of these edges over the old
             rows W (`controller_evaluate_mixed` on a graph with the n_a appended).  n_{a_0} takes n's index and the others are appended,
             and edges into n (mixture members naming n too) go to the mixture {n_a : c_a} -- only if `mixture_rows` verifies
             sum_a c_a X_{n_a} - W_n > tau / 2 at every state; otherwise n stays as it was.  With one action no mixture is needed.
             The graph grows by at most (distinct actions of the solution - 1) nodes per improved node: that is the bound of BPI here.
          3. `evaluate(gamma, eps)` from X (W on the old nodes, X_{n_a} on the new), with its certificate.
          4. Only the nodes reachable from the argmax nodes of b0 and `beliefs`, through edges and mixture members, are kept
             (`reachable_nodes`, `compact_graph`).

        Why the bound does not fall: old nodes keep W, and an edge n -> mixture whose row is >= W_n + tau / 2 only raises (T' X)_p, by
        non-negative RTO and monotone rounding.  Each n_a's edges name old rows, or improved nodes' mixtures that lie above them.  So
        X <= T' X in exact arithmetic, the new controller's value is >= X, and at every belief max_n X_n . b >= the old value.  The
        certificate of `evaluate` absorbs rounding, so what a caller can see is at most a fall by its shift.

        Stats per iteration: nodes_before, nodes_after, improved, not_improvable, budget, numerical, failed (improvable but not
        verified), unchanged (improvable, but the LP's solution is the node itself: its own action on its own edges, which only the start
        row would change; such nodes are left as they are and do not count as improved), mixtures, nnz, lp_rounds, max_columns, pivots, pool_rows, value_b0 (certified), shift and seconds {lp, select, assemble,
        build, evaluate, prune}.  An iteration that improves no node returns the graph unchanged and ends the loop.
        """
        self._require_rows()
        if self.gamma is None:
            raise ValueError('bounded_improve needs the gamma of evaluate: call evaluate(gamma) first')
        m, gamma = self.model, self.gamma
        dev = m.device
        d = dev.device
        B = belief_rows(m, m.start_probabilities)
        if beliefs is not None:
            B = torch.cat([B, belief_rows(m, beliefs)])
        pg, all_stats = self, []
        for _ in range(int(iterations)):
            W, N = pg.rows, len(pg)
            act = torch.as_tensor(pg.actions, dtype=torch.int32, device=d)
            succ = torch.as_tensor(pg.successors, dtype=torch.int32, device=d).contiguous()
            own = dev.controller_evaluate_mixed(W, gamma, act, succ, pg.mixtures or NO_MIXTURES, float('inf'), 1)[0]
            tau = 1e-9 * max(1.0, float(torch.max(torch.abs(W))), float(torch.max(torch.abs(own))))
            sol = bpi_lps(dev, W, own, gamma, tau)
            sec = dict(sol['seconds'])
            t0 = time.perf_counter()
            status = sol['status']
            nxt, splits, ok, unchanged = pg._bpi_start_graph(sol, tau)
            st = dict(nodes_before=N, improved=len(ok), not_improvable=int(np.sum(status == 1)), budget=int(np.sum(status == 3)),
                      numerical=int(np.sum(status == 4)), failed=len(splits) - len(ok), unchanged=unchanged,
                      lp_rounds=sol['stats']['rounds'], max_columns=sol['stats']['max_columns'], pivots=sol['stats']['pivots'],
                      pool_rows=sol['stats']['pool_rows'])
            if nxt is None:
                sec.update(build=time.perf_counter() - t0, evaluate=0.0, prune=0.0)
                st.update(nodes_after=N, mixtures=0 if pg.mixtures is None else len(pg.mixtures[0]) - 1,
                          nnz=0 if pg.mixtures is None else len(pg.mixtures[1]), value_b0=float(pg.value(B[:1])[0][0]), shift=0.0,
                          seconds=sec)
                all_stats.append(st)
                break
            sec['build'] = time.perf_counter() - t0
            t0 = time.perf_counter()
            rows, hist = nxt.evaluate(gamma, eps)
            sec['evaluate'] = time.perf_counter() - t0
            t0 = time.perf_counter()
            roots = dev.max_values(B, rows)[1].cpu().numpy()
            seen = reachable_nodes(nxt.successors, roots, nxt.mixtures)
            keep, k_act, k_succ, k_mix = compact_graph(nxt.actions, nxt.successors, np.where(seen, np.arange(len(nxt)), -1), nxt.mixtures)
            pg = PolicyGraph(m, k_act, k_succ, rows=rows[torch.as_tensor(keep, device=d)], mixtures=k_mix)
            pg.gamma = gamma
            sec['prune'] = time.perf_counter() - t0
            st.update(nodes_after=len(pg), mixtures=0 if k_mix is None else len(k_mix[0]) - 1, nnz=0 if k_mix is None else len(k_mix[1]),
                      value_b0=float(pg.value(B[:1])[0][0]), shift=hist.shift, seconds=sec)
            all_stats.append(st)
        return pg, all_stats

    def _bpi_start_graph(self, sol: dict, tau: float) -> tuple:
        """
        Steps 2 of `bounded_improve` on the LP solutions `sol` of `bpi_lps`: returns (the improved graph without rows and with `_initial`
        = X, or None when no node is improved; {n: split} of the improvable nodes; the verified nodes; the nodes whose LP solution is
        the node itself).  A node is improvable when its LP stopped optimal or at the budget with u < -tau; a split that plays the
        node's own action on the node's own edges (its solution is its own column) changes nothing and is left out.
        """
        m, gamma, W, N = self.model, self.gamma, self.rows, len(self)
        dev, d = m.device, m.device.device
        status = sol['status']
        improvable = np.flatnonzero(((status == 2) | (status == 3)) & (sol['u'] < -tau))
        splits, unchanged = {}, 0
        for n in improvable.tolist():
            cols, columns = sol['columns'][n], []
            for c in cols[cols > -2].tolist():
                t = sol['tuples'][c] if c >= 0 else None
                columns.append((int(self.actions[n]), self.successors[n]) if c == -1 else (int(t[0]), t[1:]))
            sp = bpi_split(columns, sol['lam'][n][:len(columns)], N, self.mixtures)
            if len(sp) == 1 and sp[0][0] == self.actions[n] and all(
                    np.array_equal(nodes, own[0]) and np.array_equal(w, own[1])
                    for (nodes, w), own in zip(sp[0][2], (combine_members(*successor_distribution(int(e), N, self.mixtures))
                                                          for e in self.successors[n]))):
                unchanged += 1
                continue
            splits[n] = sp
        if not splits:
            return None, splits, [], unchanged
        a_i, s_i, mix_i, pos_i = bpi_assemble(self.actions, self.successors, self.mixtures, splits, redirect=False)
        X0 = torch.cat([W, torch.zeros((len(a_i) - N, W.shape[1]), dtype=torch.float64, device=d)])
        Xi = dev.controller_evaluate_mixed(X0, gamma, a_i, s_i, mix_i or NO_MIXTURES, float('inf'), 1)[0]
        order = sorted(splits)
        off = np.concatenate([[0], np.cumsum([len(splits[n]) for n in order])]).astype(np.int64)
        members = np.asarray([pos_i[(n, j)] for n in order for j in range(len(splits[n]))], np.int64)
        weights = np.asarray([c for n in order for _, c, _ in splits[n]], np.float64)
        Z = mixture_rows(Xi, (off, members, weights))
        good = ((Z - W[torch.as_tensor(order, device=d)]) > tau / 2).all(dim=1).cpu().numpy()
        ok = [n for n, g in zip(order, good.tolist()) if g]
        if not ok:
            return None, splits, ok, unchanged
        a_f, s_f, mix_f, pos_f = bpi_assemble(self.actions, self.successors, self.mixtures, {n: splits[n] for n in ok}, redirect=True)
        X = torch.cat([W, torch.zeros((len(a_f) - N, W.shape[1]), dtype=torch.float64, device=d)])
        dst, src = zip(*[(k, pos_i[key]) for key, k in pos_f.items()])
        X[torch.as_tensor(dst, device=d)] = Xi[torch.as_tensor(src, device=d)]
        nxt = PolicyGraph(m, a_f, s_f, mixtures=mix_f)
        nxt._initial = X
        return nxt, splits, ok, unchanged

    def prune_dominated(self) -> 'PolicyGraph':
        """
        The graph without its pointwise-dominated nodes: a new PolicyGraph with the kept rows and `gamma`; this graph is not changed.

        Node i is dropped when some node j has W_j >= W_i at every state (`pbvi_dominating_row`: the smallest such j != i, and when j > i
        it must also be larger somewhere, so equal rows keep their first copy and witness chains cannot cycle; a row with a NaN is never a
        witness and never has one), and every edge to i goes to the kept node at the end of its witness chain (`redirect_dominated`).
        The RTO weights are non-negative, so every predecessor p sees a successor row that is at least as large:
        (T_new W)_p >= (T_old W)_p >= W_p, and no other row or entry changes.  The certificate W <= T_pi W therefore still holds and the
        kept rows need no re-evaluation.  max_n W_n . b is unchanged at every belief, bitwise in FP64: `max_values` sums every row in the
        same order with b >= 0, and rounded products, sums and FMAs are monotone in each argument, so the computed value of W_j is >= that
        of W_i.  In a graph with mixtures the members of every mixture go along the witness chains too (a mixture row can only rise,
        entry by entry), and only the mixtures that some kept edge references are kept.
        """
        W = self._require_rows()
        witness = self.model.device.dominating_row(W).cpu().numpy()
        if self.mixtures is None:
            keep, act, succ = redirect_dominated(self.actions, self.successors, witness)
            mix = None
        else:
            keep, act, succ, mix = compact_graph(self.actions, self.successors, resolve_witnesses(witness), self.mixtures)
        pg = PolicyGraph(self.model, act, succ, rows=W[torch.as_tensor(keep, device=W.device)], mixtures=mix)
        pg.gamma = self.gamma
        return pg

    def prune_lp(self) -> 'PolicyGraph':
        """
        The graph without the nodes that a convex combination of other nodes dominates: a new PolicyGraph with mixtures, the kept rows,
        `gamma` and `prune_stats`; this graph is not changed.  Needs rows (an evaluated graph) and a graph without mixtures.

          1. `prune_dominated()`: `pbvi_prune_lp` needs pairwise distinct rows, and pointwise pruning leaves no two equal rows.
          2. `pbvi_prune_lp_certificates` on the rows: node i is pruned when a convex combination lambda of other rows exceeds W_i by more
             than tau = 1e-9 * max(1, max |W|) at every state (verified in FP64), and lambda comes back with it.
          3. `resolve_certificates`: lambda's weight on pruned nodes is substituted by their own combinations until it is negligible; small
             weights are dropped and the rest renormalised: a mixture of kept nodes per pruned node.
          4. Each mixture is verified on the device: Z_i = `mixture_rows` (the arithmetic of the mixture phase of the sweeps) must satisfy
             Z_i[s] - W_i[s] > tau / 2 at every state.  A node that fails is kept with its own edges; the others stay valid, because each
             mixture is verified on its own and names kept nodes only.
          5. Every edge into a pruned node goes to its mixture (successor entry N' + m); only mixtures that some edge references are stored.

        Why nothing needs re-evaluation: the RTO weights are non-negative and the computed Z_i >= W_i entry by entry, and rounded products
        and sums are monotone in each argument, so every predecessor p sees (T' W)_p >= (T W)_p >= W_p in the sweep's own arithmetic: the
        certificate W <= T_pi W survives.  The value is bitwise unchanged: tau / 2 is far above the rounding of a dot product (even at
        S = 22 021, FP64 rounding of b . W is below 1e-11 relative), and Z_i is a convex combination of kept rows, so some kept row beats
        W_i . b at every belief b and a pruned row never attains max_n W_n . b; that maximum, over the same kept rows in the same order, is
        bitwise the same at every belief, with the same best node.  An `evaluate` afterwards starts from rows that satisfy X <= T_pi' X,
        so its certified value can only rise, up to its own shift.

        `prune_stats`: nodes, after_dominated, nodes_after, mixtures, nnz, lp_counts (kept at a corner, kept by an LP witness, pruned, kept
        undecided), lp_stats (`prune_lp_stats`), failed (pruned by the LP but not verified) and seconds.
        """
        t0 = time.perf_counter()
        self._require_rows()
        if self.mixtures is not None:
            raise ValueError('prune_lp needs a graph without mixtures')
        dev = self.model.device
        pd = self.prune_dominated()
        W = pd.rows
        N = len(pd)
        keep, _, counts, cidx, cw = dev.prune_lp_certificates(W)
        lp_stats = dev.prune_lp_stats()
        pruned = keep.cpu().numpy() == 0
        res = resolve_certificates(pruned, cidx.cpu().numpy(), cw.cpu().numpy())
        cand = sorted(res)
        ok = np.zeros(0, dtype=bool)
        if cand:
            off = np.concatenate([[0], np.cumsum([len(res[i][0]) for i in cand])]).astype(np.int64)
            table = (off, np.concatenate([res[i][0] for i in cand]), np.concatenate([res[i][1] for i in cand]))
            tau = 1e-9 * max(1.0, float(torch.max(torch.abs(W))))
            Z = mixture_rows(W, table)
            ok = ((Z - W[torch.as_tensor(cand, device=W.device)]) > tau / 2).all(dim=1).cpu().numpy()
        redirect = np.arange(N, dtype=np.int64)
        good = [i for i, v in zip(cand, ok.tolist()) if v]
        if good:
            redirect[good] = N + np.flatnonzero(ok)
            kept, act, succ, mix = compact_graph(pd.actions, pd.successors, redirect, table, np.arange(N))
        else:
            kept, act, succ, mix = np.arange(N), pd.actions, pd.successors, None
        pg = PolicyGraph(self.model, act, succ, rows=W[torch.as_tensor(kept, device=W.device)], mixtures=mix)
        pg.gamma = self.gamma
        pg.prune_stats = dict(nodes=len(self), after_dominated=N, nodes_after=len(pg), mixtures=0 if mix is None else len(mix[0]) - 1,
                              nnz=0 if mix is None else len(mix[1]), lp_counts=counts.tolist(), lp_stats=lp_stats,
                              failed=int(pruned.sum()) - len(good), seconds=time.perf_counter() - t0)
        return pg

    def _require_rows(self) -> torch.Tensor:
        if self.rows is None:
            raise ValueError('the graph has no rows yet: call evaluate(gamma) first')
        return self.rows

    @property
    def value_function(self) -> ValueFunction:
        """The node rows as a ValueFunction with the node actions (e.g. for `UpperBound.gap`)."""
        if self._value_function is None:
            self._value_function = ValueFunction(self.model, self._require_rows(), self.actions)
        return self._value_function

    def value(self, beliefs) -> tuple:
        """(max_n W_n . b [n] CUDA float64, best start node [n] CUDA int32) for every belief."""
        return self.model.device.max_values(belief_rows(self.model, beliefs), self._require_rows())

    # ---- validation by simulation --------------------------------------------------------------------------------------------
    def simulate(self, n: int, max_steps: int, seed: int, start_belief=None) -> np.ndarray:
        """
        Discounted returns [n] of `n` host-side roll-outs of `max_steps` steps with the discount of the last `evaluate`.  Start states are
        drawn from the belief (default b0), and every agent starts in the best node for it.  Each step collects Rbar[s, a_node], draws
        (o, r) jointly from RTO[s, a_node, :, :], then moves s <- reach[s, a, r] and node <- sigma(node, o).  A validation tool, not a
        hot path: NumPy, vectorised over agents.  Raises ValueError when an RTO row does not sum to 1 (within 1e-9).
        In a graph with mixtures every step draws one more uniform per agent (after the observation's), and an agent whose edge leads to
        mixture m moves to the first member k whose cumulative weight exceeds it; a graph without mixtures draws nothing more.
        """
        self._require_rows()
        if self.gamma is None:
            raise ValueError('simulate discounts with the gamma of evaluate: call evaluate(gamma) first')
        m = self.model
        reach = np.asarray(m.reachable_states, dtype=np.int64)
        rto = np.asarray(m.reachable_transitional_observation_table, dtype=np.float64)
        rbar = np.asarray(m.expected_rewards_table, dtype=np.float64)
        S, A, O, R = rto.shape
        if not np.all(np.abs(rto.sum(axis=(2, 3)) - 1.0) <= 1e-9):
            raise ValueError('simulate needs RTO rows that sum to 1 (a model with end states or leaking mass cannot be rolled out)')
        b = belief_rows(m, m.start_probabilities if start_belief is None else start_belief)[:1]
        node0 = int(self.value(b)[1][0])
        p = b[0].cpu().numpy()
        rng = np.random.default_rng(seed)
        s = rng.choice(S, size=n, p=p / p.sum())
        node = np.full(n, node0, dtype=np.int64)
        cdf = np.cumsum(rto.reshape(S, A, O * R), axis=2)
        N = len(self)
        if self.mixtures is not None:
            off, members, w = self.mixtures
            mix_of = np.repeat(np.arange(len(off) - 1), np.diff(off))
            # member k of mixture m covers cumulative weights up to m + sum_{k' <= k} w_k' (within the mixture): one sorted key array
            key = mix_of + np.concatenate([np.cumsum(w[off[m]:off[m + 1]]) for m in range(len(off) - 1)])
        ret = np.zeros(n)
        disc = 1.0
        for _ in range(max_steps):
            a = self.actions[node]
            ret += disc * rbar[s, a]
            u = rng.random(n)
            k = np.minimum((cdf[s, a] <= u[:, None]).sum(axis=1), O * R - 1)
            o, r = k // R, k % R
            s = reach[s, a, r]
            node = self.successors[node, o]
            if self.mixtures is not None:
                u2 = rng.random(n)
                mx = np.flatnonzero(node >= N)
                m = node[mx] - N
                k = np.searchsorted(key, m + u2[mx], side='right')
                node[mx] = members[np.clip(k, off[m], off[m + 1] - 1)]
            disc *= self.gamma
        return ret

    def outcomes(self, max_steps: int, beliefs=None, start_nodes=None, gamma=None) -> ControllerOutcomes:
        """
        Exact outcomes of the controller's runs under the reference's termination rule (`Simulation.run_action`): a run starts in a state
        s and a node n, each step plays a = a_n, collects Rbar[s, a], draws (o, r) from RTO[s, a, :, :] and moves to reach[s, a, r] and
        sigma(n, o).  It stops after a step that lands in one of the model's `end_states` or plays one of its `end_actions`; that step's
        reward counts, nothing after it does, and a run that starts in an end state still takes its first step.  With T the stopping step
        and H = `max_steps`, returns (`ControllerOutcomes`) P(T <= H), E[min(T, H)] and the discounted return
        G = E[sum_{t < min(T, H)} gamma^t r_t] at each query pair, the same after every k <= H, and the rows over every (node, state).
        No sampling: `pbvi_controller_outcomes` runs the H steps of the three recursions over (node, state) in one persistent launch
        (`pbvi_controller_outcomes_mixed` for a graph with mixtures: a mixture successor contributes the mixture of its members' rows).

        G starts its discount at 1 (gamma^0 on the first reward); the average discounted reward the reference's simulations print starts
        it at gamma, so it is gamma * G.  With gamma = 1 and a finite H, G is the reference's average total reward.

        Query pairs: the rows of `beliefs` (default: b0) with `start_nodes` (default: the best node at each belief, as `simulate` starts).
        `gamma` defaults to the gamma of the last `evaluate` and may be anywhere in (0, 1].  Raises ValueError when there is no gamma, gamma
        is outside (0, 1], max_steps < 0, the graph has no rows and no `start_nodes` are given, or an RTO row does not sum to 1 within
        1e-9 (as `simulate`); non-finite beliefs are rejected by `belief_rows`.
        """
        gamma = self.gamma if gamma is None else gamma
        if gamma is None:
            raise ValueError('outcomes needs a gamma: pass one or call evaluate(gamma) first')
        gamma = float(gamma)
        if not 0.0 < gamma <= 1.0:
            raise ValueError('gamma must lie in (0, 1]')
        if int(max_steps) != max_steps or max_steps < 0:
            raise ValueError('max_steps must be an integer >= 0')
        max_steps = int(max_steps)
        m = self.model
        rto = np.asarray(m.reachable_transitional_observation_table, dtype=np.float64)
        if not np.all(np.abs(rto.sum(axis=(2, 3)) - 1.0) <= 1e-9):
            raise ValueError('outcomes needs RTO rows that sum to 1 (a model with leaking mass has no run distribution)')
        if start_nodes is None and self.rows is None:
            raise ValueError('the graph has no rows to choose start nodes by: pass start_nodes or call evaluate(gamma) first')
        B = belief_rows(m, m.start_probabilities if beliefs is None else beliefs)
        if start_nodes is None:
            nodes = self.value(B)[1].cpu().numpy().astype(np.int64)
        else:
            nodes = np.asarray(start_nodes, dtype=np.int64).reshape(-1)
            if nodes.shape != (B.shape[0],):
                raise ValueError(f'start_nodes must have one node per belief row ({B.shape[0]}), got {nodes.shape[0]}')
            if nodes.size and (nodes.min() < 0 or nodes.max() >= len(self)):
                raise ValueError(f'start nodes must lie in [0, {len(self)})')
        end_state = np.zeros(m.state_count, dtype=np.uint8)
        end_state[np.asarray(m.end_states, dtype=np.int64)] = 1
        end_action = np.zeros(m.action_count, dtype=np.uint8)
        end_action[np.asarray(m.end_actions, dtype=np.int64)] = 1
        if self.mixtures is None:
            P, M, G, series = m.device.controller_outcomes(self.actions, self.successors, end_state, end_action, gamma, max_steps, B, nodes)
        else:
            P, M, G, series = m.device.controller_outcomes_mixed(self.actions, self.successors, self.mixtures, end_state, end_action, gamma,
                                                                 max_steps, B, nodes)
        return ControllerOutcomes(nodes, series.cpu().numpy(), (P, M, G), gamma, max_steps)

    # ---- persistence (pomdp-solve formats) --------------------------------------------------------------------------------
    def save(self, path: str, name: str) -> None:
        """Writes `<path>/<name>.pg`, when the graph has rows `<path>/<name>.alpha`, and when it has mixtures `<path>/<name>.mix`
        ("mixture_id k node_1 weight_1 ... node_k weight_k" per mixture).  Values and weights as %.17g: a round trip is bitwise."""
        os.makedirs(path, exist_ok=True)
        with open(os.path.join(path, name + '.pg'), 'w') as f:
            for i in range(len(self)):
                f.write(' '.join(str(int(x)) for x in (i, self.actions[i], *self.successors[i])) + '\n')
        if self.rows is not None:
            rows = self.rows.cpu().numpy()
            with open(os.path.join(path, name + '.alpha'), 'w') as f:
                for i in range(len(self)):
                    f.write(f'{int(self.actions[i])}\n' + ' '.join('%.17g' % x for x in rows[i]) + '\n\n')
        if self.mixtures is not None:
            off, members, w = self.mixtures
            with open(os.path.join(path, name + '.mix'), 'w') as f:
                for m in range(len(off) - 1):
                    pairs = ' '.join(f'{int(members[k])} {w[k]:.17g}' for k in range(off[m], off[m + 1]))
                    f.write(f'{m} {off[m + 1] - off[m]} {pairs}\n')

    @classmethod
    def load(cls, path: str, name: str, model: Model) -> 'PolicyGraph':
        """Reads what `save` wrote (the `.alpha` and `.mix` files are optional); node ids must be 0..N-1 and mixture ids 0..M-1 in order."""
        with open(os.path.join(path, name + '.pg')) as f:
            lines = [ln.split() for ln in f if ln.strip()]
        table = np.asarray([[int(x) for x in ln] for ln in lines], dtype=np.int64)
        if table.ndim != 2 or table.shape[1] != 2 + model.observation_count or not np.array_equal(table[:, 0], np.arange(len(table))):
            raise ValueError(f'{name}.pg: expected lines "id action succ_0 .. succ_{model.observation_count - 1}" with ids 0..N-1')
        rows = None
        alpha = os.path.join(path, name + '.alpha')
        if os.path.isfile(alpha):
            with open(alpha) as f:
                lines = [ln.split() for ln in f if ln.strip()]
            if len(lines) != 2 * len(table) or any(int(lines[2 * i][0]) != table[i, 1] for i in range(len(table))):
                raise ValueError(f'{name}.alpha does not match {name}.pg')
            rows = np.asarray([[float(x) for x in lines[2 * i + 1]] for i in range(len(table))], dtype=np.float64)
        mixtures = None
        mix = os.path.join(path, name + '.mix')
        if os.path.isfile(mix):
            with open(mix) as f:
                lines = [ln.split() for ln in f if ln.strip()]
            off, members, weights = [0], [], []
            for m, ln in enumerate(lines):
                if int(ln[0]) != m or len(ln) != 2 + 2 * int(ln[1]):
                    raise ValueError(f'{name}.mix: expected lines "mixture_id k node_1 weight_1 .. node_k weight_k" with ids 0..M-1')
                members += [int(x) for x in ln[2::2]]
                weights += [float(x) for x in ln[3::2]]
                off.append(len(members))
            mixtures = (np.asarray(off, dtype=np.int64), np.asarray(members, dtype=np.int64), np.asarray(weights, dtype=np.float64))
        return cls(model, table[:, 1], table[:, 2:], rows=rows, mixtures=mixtures)
