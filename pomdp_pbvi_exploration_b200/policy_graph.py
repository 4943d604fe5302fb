"""
Finite-state controllers (policy graphs) extracted from a value function, and their exact evaluation as a certified lower bound on V*.

    PolicyGraph   N nodes, node n playing action a_n and moving to node sigma(n, o) on observation o.  Its value vectors solve
                      V_n = Rbar_{a_n} + gamma * sum_o sum_r RTO[., a_n, o, r] * V_{sigma(n,o)}[reach[., a_n, r]]
                  and max_n V_n . b is the value of a policy that can be executed, hence a lower bound on V*(b) at every belief and for
                  every model, whatever the signs of its rewards.  `evaluate` iterates that fixed point on the device (one
                  persistent `pbvi_controller_evaluate` launch) and certifies the returned rows with a residual shift; `improve`
                  raises that bound by point-based policy iteration on the controller.

The file formats of `save` / `load` are pomdp-solve's: `.pg` ("id action succ_0 ... succ_{O-1}" per node) and `.alpha` (an action line, a
values line and a blank line per node).
"""
from __future__ import annotations

import os
import time

import numpy as np
import torch

from .bounds import belief_rows, certificate_contraction
from .model import Model, log
from .solver import MDPSolverHistory
from .value_function import ValueFunction


def reachable_subgraph(actions, successors, roots) -> tuple:
    """
    The part of a controller that can run from the nodes `roots`: returns (kept node indices ascending, their actions, their successors
    renumbered to positions in the kept list).  Kept nodes keep their relative order, and every successor of a kept node is kept
    (whatever the observation, an impossible one included), so the rows of the kept nodes need no re-evaluation.
    """
    act = np.asarray(actions, dtype=np.int64).reshape(-1)
    succ = np.asarray(successors, dtype=np.int64)
    seen = np.zeros(act.shape[0], dtype=bool)
    stack = sorted({int(r) for r in np.asarray(roots).reshape(-1)})
    seen[stack] = True
    while stack:
        for t in succ[stack.pop()].tolist():
            if not seen[t]:
                seen[t] = True
                stack.append(t)
    keep = np.flatnonzero(seen)
    renumber = np.full(act.shape[0], -1, dtype=np.int64)
    renumber[keep] = np.arange(len(keep))
    return keep, act[keep], renumber[succ[keep]]


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


class PolicyGraph:
    """
    A finite-state controller over `model`: `actions` [N] and `successors` [N, O] (node indices) as host int64 arrays; after `evaluate` (or
    `load` of a saved graph with rows) `rows` [N, S] is a CUDA float64 tensor of node values.  `source_rows` [N] holds, for an extracted
    graph, the row of the value function each node came from (None otherwise).
    """

    def __init__(self, model: Model, actions, successors, rows=None, source_rows=None):
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
        if succ.min() < 0 or succ.max() >= N:
            raise ValueError(f'successor nodes must lie in [0, {N})')
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
        eps * gamma / (1 - gamma) or `max_sweeps` sweeps.  Certificate, the
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
            W, changes, k = dev.controller_evaluate(W, gamma, act, succ, tol, max_sweeps)
            changes = changes.cpu().numpy().tolist()
            per_sweep = (time.perf_counter() - start) / k
            for c in changes:
                history.add(per_sweep, c, None)
            change = changes[-1]
            if change != change:
                raise ValueError('the controller iterates are not finite')
        residual = float(dev.controller_sweep(W, gamma, act, succ, want_stats=True)[1][1])
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
            left = float(dev.controller_sweep(W, gamma, act, succ, want_stats=True)[1][1])
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
        seconds {select, assemble, dominance, evaluate, prune}.
        """
        self._require_rows()
        if self.gamma is None:
            raise ValueError('improve needs the gamma of evaluate: call evaluate(gamma) first')
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
            disc *= self.gamma
        return ret

    # ---- persistence (pomdp-solve formats) --------------------------------------------------------------------------------
    def save(self, path: str, name: str) -> None:
        """Writes `<path>/<name>.pg` and, when the graph has rows, `<path>/<name>.alpha` (values as %.17g: a round trip is bitwise)."""
        os.makedirs(path, exist_ok=True)
        with open(os.path.join(path, name + '.pg'), 'w') as f:
            for i in range(len(self)):
                f.write(' '.join(str(int(x)) for x in (i, self.actions[i], *self.successors[i])) + '\n')
        if self.rows is not None:
            rows = self.rows.cpu().numpy()
            with open(os.path.join(path, name + '.alpha'), 'w') as f:
                for i in range(len(self)):
                    f.write(f'{int(self.actions[i])}\n' + ' '.join('%.17g' % x for x in rows[i]) + '\n\n')

    @classmethod
    def load(cls, path: str, name: str, model: Model) -> 'PolicyGraph':
        """Reads what `save` wrote (the `.alpha` file is optional); node ids must be 0..N-1 in order."""
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
        return cls(model, table[:, 1], table[:, 2:], rows=rows)
