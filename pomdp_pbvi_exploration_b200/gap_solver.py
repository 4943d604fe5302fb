"""
Gap-driven trials from b0 (HSVI2's exploration, Smith & Simmons 2005) between the certified bounds of this package, stopping at a certified
optimality gap at b0:

    lower   an append-only `PolicyGraph` (start: the blind controller, evaluated), raised by point-based controller backups at trial beliefs
    upper   an `UpperBound` (start: the FIB bound), lowered by point-based upper-bound backups at trial beliefs

A round runs K trials at once, one `pbvi_gap_trial_step` call per depth level (`DeviceModel.gap_trial_step`), then backs both bounds up
level by level, deepest first.  When upper(b0) - lower(b0) <= target_gap the controller is certified (`PolicyGraph.evaluate` from its
rows) and pruned to what b0's best node reaches; the solve ends when the certified gap is within the target.
"""
from __future__ import annotations

import time

import numpy as np
import torch

from .bounds import FIB_Solver, UpperBound, belief_rows, certificate_contraction
from .model import Model, log
from .policy_graph import PolicyGraph, backup_tuples, match_tuples, node_index, reachable_subgraph


class GapSolverHistory:
    """
    What a `GapSolver.solve` did:
      reached        True when the certified gap at b0 is within target_gap
      lower, upper   the certified bounds at b0 of the returned graph and upper bound
      shift          the certificate shift of the last `evaluate`
      rounds         one dict per round: round, seconds (wall time since the start), upper_b0, lower_b0 (max_n X_n . b0 of the
                     uncertified rows), nodes, stored_pairs, depths (per trial: depth of its last belief), phase_seconds {descent, lower,
                     upper, certify} and, in the rounds that certified, certified_lower / certified_upper
      seconds        wall time of the whole solve
      uncertified    the append-only controller with its rows X before the last certificate (X <= T_pi X)
    """

    def __init__(self, gamma: float, target_gap: float, trials: int, max_depth: int, seed: int):
        self.gamma, self.target_gap, self.trials, self.max_depth, self.seed = gamma, target_gap, trials, max_depth, seed
        self.reached = False
        self.lower = self.upper = self.shift = None
        self.rounds = []
        self.seconds = 0.0
        self.uncertified = None

    @property
    def gap(self) -> float:
        return self.upper - self.lower


class _AppendOnlyGraph:
    """
    The solver's lower bound: a controller whose nodes are only ever appended.  rows X [N, S] start certified (X <= T_pi X); a backup
    at beliefs B appends, for every backup tuple t_b = (a*, v*[b, a*, :]) against X that no node plays yet, the node t_b with the row
    Y = `backup_assemble(X, t_b)`.  Its successors are old nodes, whose rows and transitions do not change, so Y = (T_pi X)_new and
    the old entries of T_pi X stay as they were: X <= T_pi X holds after every backup, and max_n X_n . b <= V*(b) in exact arithmetic.
    """

    def __init__(self, model: Model, gamma: float, actions, successors, rows: torch.Tensor):
        self.model, self.gamma = model, gamma
        self.actions = list(np.asarray(actions, dtype=np.int64))
        self.successors = [np.asarray(s, dtype=np.int64) for s in successors]
        self.node_of = node_index(self.actions, self.successors)
        self.n = rows.shape[0]
        self._X = torch.empty((max(64, 2 * self.n), model.state_count), dtype=torch.float64, device=rows.device)
        self._X[:self.n] = rows

    @property
    def rows(self) -> torch.Tensor:
        return self._X[:self.n]

    def backup(self, beliefs: torch.Tensor) -> int:
        dev = self.model.device
        _, new_t = match_tuples(self.node_of, backup_tuples(dev, beliefs, self.rows, self.gamma))
        k = len(new_t)
        if k == 0:
            return 0
        Y = dev.backup_assemble(self.rows, self.gamma, new_t[:, 0], new_t[:, 1:])
        if self.n + k > self._X.shape[0]:
            grown = torch.empty((2 * (self.n + k), self._X.shape[1]), dtype=torch.float64, device=self._X.device)
            grown[:self.n] = self.rows
            self._X = grown
        self._X[self.n:self.n + k] = Y
        for t in new_t:
            self.node_of[tuple(t.tolist())] = len(self.actions)
            self.actions.append(int(t[0]))
            self.successors.append(t[1:].copy())
        self.n += k
        return k

    def certify(self, b0: torch.Tensor, eps: float) -> tuple:
        """(certified PolicyGraph pruned to what b0's best node reaches, its value at b0, the certificate shift)."""
        act, succ = np.asarray(self.actions), np.stack(self.successors)
        pg = PolicyGraph(self.model, act, succ)
        pg._initial = self.rows.clone()
        rows, hist = pg.evaluate(self.gamma, eps)
        roots = self.model.device.max_values(b0, rows)[1].cpu().numpy()
        keep, k_act, k_succ = reachable_subgraph(act, succ, roots)
        out = PolicyGraph(self.model, k_act, k_succ, rows=rows[torch.as_tensor(keep, device=rows.device)])
        out.gamma = self.gamma
        return out, float(out.value(b0)[0][0]), hist.shift


def _distinct_rows(dev, rows: torch.Tensor) -> torch.Tensor:
    """The rows in order of first occurrence without bytewise repeats (128-bit row keys, every key match confirmed)."""
    keys = dev.row_hash(rows).cpu().numpy()
    first, keep = {}, []
    for i, key in enumerate(map(tuple, keys.tolist())):
        j = first.get(key)
        if j is None:
            first[key] = i
            keep.append(i)
        elif not torch.equal(rows[i], rows[j]):
            keep.append(i)
    return rows[torch.as_tensor(keep, device=rows.device)] if len(keep) < rows.shape[0] else rows


class GapSolver:
    """
    Solve until upper(b0) - lower(b0) <= target_gap, with certified bounds at both ends.

    One round:
      1. K = `trials` trials start at b0.  At depth t every live trial takes one `gap_trial_step` with theta_t = target_gap * gamma^-t:
         a* maximises the upper-bound Q-value, o* has the largest weighted excess P(o|b,a*) * (U - L - theta_t) (trial 0 always; trials
         1..K-1 draw o* with weights equal to the positive excesses, from uniforms of np.random.default_rng(seed) drawn K-1 per level in
         trial order).  A trial ends when no excess is positive; beliefs of depth max_depth are not visited.
      2. Deepest level first, the level's distinct beliefs get a lower backup (new controller nodes, see `_AppendOnlyGraph`) and then
         `UpperBound.improve`.
      3. When upper(b0) - max_n X_n . b0 <= target_gap the controller is certified (`PolicyGraph.evaluate` from X, then
         `reachable_subgraph`); the solve ends if the certified gap is within the target.
    `max_rounds` and `time_limit` (seconds, checked before each round) also end a solve; the returned graph is certified either way.
    Upper(b0) never rises (stored upper values only decrease) and the uncertified lower(b0) never falls (nodes are only appended).
    The solve is deterministic for a given seed; with trials = 1 the seed is not used.
    """

    def __init__(self, gamma: float, target_gap: float, trials: int = 8, max_depth: int = 200, seed: int = 0):
        if not target_gap > 0.0:
            raise ValueError('target_gap must be positive')
        if trials < 1 or max_depth < 1:
            raise ValueError('trials and max_depth must be at least 1')
        self.gamma, self.target_gap, self.trials, self.max_depth, self.seed = float(gamma), float(target_gap), int(trials), int(max_depth), seed

    def solve(self, model: Model, max_rounds: int = 100, time_limit: float | None = None, lower: PolicyGraph | None = None,
              upper: UpperBound | None = None, eps: float = 1e-6, print_progress: bool = False) -> tuple:
        """Returns (certified PolicyGraph, UpperBound, GapSolverHistory).  `lower`: an evaluated PolicyGraph to start from (default: the
        blind controller); `upper`: an UpperBound with this gamma (default: the FIB bound, eps 1e-6).  `eps` is the evaluation
        tolerance of the certificates.  gamma' >= 1 raises ValueError."""
        gamma, target, K = self.gamma, self.target_gap, self.trials
        if not 0.0 < gamma < 1.0:
            raise ValueError('gamma must lie in (0, 1)')
        certificate_contraction(model, gamma, 'controller')
        t_start = time.perf_counter()
        dev = model.device
        b0 = belief_rows(model, model.start_probabilities)[:1]
        S = model.state_count
        if lower is None:
            lower = PolicyGraph.blind(model)
            lower.evaluate(gamma, eps)
        elif lower.rows is None or lower.gamma != gamma:
            raise ValueError('lower must be a PolicyGraph evaluated with the solver gamma')
        if upper is None:
            upper = UpperBound(model, FIB_Solver(gamma=gamma, eps=1e-6).solve(model, print_progress=False)[0], gamma)
        elif upper.gamma != gamma:
            raise ValueError('upper must be an UpperBound with the solver gamma')
        graph = _AppendOnlyGraph(model, gamma, lower.actions, lower.successors, lower.rows)
        rng = np.random.default_rng(self.seed)
        history = GapSolverHistory(gamma, target, K, self.max_depth, self.seed)
        certified, cert_at = None, -1                  # the last certified graph and the node count it was made from

        def sync_time():
            torch.cuda.synchronize(dev.device)
            return time.perf_counter()

        for rnd in range(int(max_rounds)):
            if time_limit is not None and time.perf_counter() - t_start >= time_limit:
                break
            sec = dict(descent=0.0, lower=0.0, upper=0.0, certify=0.0)
            # ---- 1. descent ----
            t0 = sync_time()
            cur = b0.expand(K, S).contiguous()
            ids = np.arange(K)
            depths = np.zeros(K, dtype=np.int64)
            levels = []
            for t in range(self.max_depth):
                levels.append(cur)
                if t == self.max_depth - 1:
                    break
                draws = rng.random(K - 1)
                u = np.concatenate([[-1.0], draws])[ids]
                theta = target * gamma ** -t
                res, nxt = [], []
                i0 = 0
                while i0 < len(ids):
                    nc = upper._chunk(len(ids) - i0)
                    idx, val, count, dot, vals, n_ub = upper._lists()
                    out, nb = dev.gap_trial_step(cur[i0:i0 + nc], graph.rows, upper._F, gamma, upper.corner_values, idx, val, count, dot,
                                                 vals, n_ub, theta, u[i0:i0 + nc])
                    res.append(out.cpu().numpy())
                    nxt.append(nb)
                    i0 += nc
                res = np.concatenate(res)
                go = res[:, 1] >= 0
                if not go.any():
                    break
                ids = ids[go]
                depths[ids] = t + 1
                cur = torch.cat(nxt)[torch.as_tensor(np.flatnonzero(go), device=cur.device)].contiguous()
            sec['descent'] = sync_time() - t0
            # ---- 2. backups, deepest level first ----
            for B in reversed(levels):
                Bu = _distinct_rows(dev, B)
                t0 = time.perf_counter()
                graph.backup(Bu)
                t1 = sync_time()
                upper.improve(Bu)
                t2 = sync_time()
                sec['lower'] += t1 - t0
                sec['upper'] += t2 - t1
            up_b0 = float(upper.evaluate(b0)[0])
            lo_b0 = float(dev.max_values(b0, graph.rows)[0][0])
            rec = dict(round=rnd, upper_b0=up_b0, lower_b0=lo_b0, nodes=graph.n, stored_pairs=len(upper), depths=depths.tolist())
            # ---- 3. certificate ----
            if up_b0 - lo_b0 <= target:
                t0 = time.perf_counter()
                certified, history.lower, history.shift = graph.certify(b0, eps)
                cert_at = graph.n
                history.upper = up_b0
                sec['certify'] = sync_time() - t0
                rec.update(certified_lower=history.lower, certified_upper=up_b0)
            rec.update(phase_seconds=sec, seconds=time.perf_counter() - t_start)
            history.rounds.append(rec)
            if print_progress:
                log(f'GapSolver round {rnd}: upper {up_b0:.6g}, lower {lo_b0:.6g}, {graph.n} nodes, {len(upper)} stored pairs, '
                    f'max depth {int(depths.max())}')
            if certified is not None and cert_at == graph.n and history.upper - history.lower <= target:
                history.reached = True
                break
        if certified is None or cert_at != graph.n or history.upper != float(upper.evaluate(b0)[0]):
            certified, history.lower, history.shift = graph.certify(b0, eps)
            history.upper = float(upper.evaluate(b0)[0])
        history.reached = history.upper - history.lower <= target
        history.uncertified = PolicyGraph(model, np.asarray(graph.actions), np.stack(graph.successors), rows=graph.rows)
        history.uncertified.gamma = gamma
        history.seconds = time.perf_counter() - t_start
        if print_progress:
            log(f'GapSolver: certified [{history.lower:.6g}, {history.upper:.6g}] at b0, gap {history.gap:.3g} '
                f'(target {target:.3g}{", reached" if history.reached else ""}), {len(certified)} nodes')
        return certified, upper, history
