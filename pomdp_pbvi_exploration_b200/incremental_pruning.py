"""
Exact value iteration by incremental pruning (Cassandra, Littman & Zhang 1997; the default algorithm of pomdp-solve), on the device.

One epoch computes V' = H V exactly, as a set of alpha vectors.  For every action a:

    Gamma^{a,o} = { gamma * sum_r RTO[:,a,o,r] * alpha_v[reach[:,a,r]] : v in V }          (`DeviceModel.ip_project`)
    acc = prune(Gamma^{a,0});  acc = prune(acc (+) prune(Gamma^{a,o})) for o = 1 .. O-1      (`DeviceModel.ip_cross_sum`)

where the last cross sum also adds Rbar[:,a], and then V' = prune(union over a, in action order).  `prune` removes the rows that another row
dominates pointwise (`dominating_row`: this also removes exact duplicates, keeping the first) and then the rows with an LP certificate
(`prune_lp`).  Both rules only remove a row that other kept rows beat at every belief, so max over the kept rows equals max over every
candidate at every belief: there is no epsilon-pruning.  Each row carries its tuple (a, v_0 .. v_{O-1}) into the rows of V, and is bitwise
`backup_assemble(V, a, v)`: the projections are alpha_a_entry's terms and the cross sums its left fold over observations.  Rows keep
candidate order (i-major, j-minor within a cross sum, actions ascending in the union), so a solve is bitwise repeatable.
"""
from __future__ import annotations

import time

import numpy as np
import torch

from .bounds import certificate_contraction
from .model import Model, log
from .value_function import ValueFunction

ULP = 2.0 ** -52
LP_COMPETITORS = 64                 # pbvi_ip_residual_lp's largest competitor set (J of the bound u)


def tuple_product(x_tuples: np.ndarray, g_ids: np.ndarray) -> np.ndarray:
    """Tuples of the rows of a cross sum x (+) g in `ip_cross_sum`'s order (i-major, j-minor): [nx * ng, k + 1], the k columns of x_i's
    tuple followed by g_j's id."""
    nx, ng = x_tuples.shape[0], g_ids.shape[0]
    return np.concatenate([np.repeat(x_tuples, ng, axis=0), np.tile(g_ids, nx)[:, None]], axis=1)


def rounding_allowance(O: int, R: int, rbar_max: float, gamma: float, rto_mass: float, alpha_max: float, new_max: float) -> tuple:
    """(rho_rows, rho_u) of the certificate in `IncrementalPruning_Solver.solve`: rho_rows bounds |computed row - exact row| of every row of
    H V built from rows with max |alpha| = alpha_max, rho_u the rounding of the FP64 re-check behind a residual bound u (rows of H V with
    max |y| = new_max tested against rows with max |x| = alpha_max)."""
    rho_rows = (O * R + 2) * ULP * (rbar_max + gamma * rto_mass * alpha_max)
    rho_u = (LP_COMPETITORS + 2) * ULP * (new_max + alpha_max)
    return rho_rows, rho_u


class IncrementalPruningHistory:
    """
    What an `IncrementalPruning_Solver.solve` did:
      epochs     one dict per completed epoch: epoch, rows (|V'|), fold_candidates (per action, the largest candidate set of its fold),
                 union_candidates, dropped_pointwise, dropped_lp, undecided (rows the LP prune kept without a decision), prune_lp_stats
                 (summed over the epoch's prune calls), residual_stats, max_u, e, shift (None without a contraction), seconds {project,
                 cross_sum, pointwise, lp, residual}, elapsed (wall time since the start of the solve)
      stopped    'target', 'horizon', 'time' or 'candidates'
      e, shift   the certificate of the returned value function (None when no epoch completed; shift None without a contraction)
      tuples     [n, 1 + O] int64: (a, v_0 .. v_{O-1}) of every returned row, v into `previous`
      previous   [m, S] CUDA float64: the rows the last epoch backed up
      seconds    wall time of the solve
    """

    def __init__(self, gamma: float, eps: float):
        self.gamma, self.eps = gamma, eps
        self.epochs = []
        self.stopped = None
        self.e = self.shift = None
        self.tuples = None
        self.previous = None
        self.seconds = 0.0

    def comparable(self) -> list:
        """The epochs without their timings (what two solves of one problem share bit for bit)."""
        return [{k: v for k, v in ep.items() if k not in ('seconds', 'elapsed')} for ep in self.epochs]


class _Candidates(Exception):
    pass


class IncrementalPruning_Solver:
    """
    Exact value iteration by incremental pruning (see the module docstring), with a certified distance to V* at every belief.

    Certificate.  After an epoch V -> V', `pbvi_ip_residual_lp` bounds, for every row y_i of V', delta_i = max_b min_j b . (y_i - x_j) over
    the rows x_j of V by a verified u_i >= delta_i, so max_i u_i >= max_b (V'(b) - V(b)) up to the rounding of u's re-check.  Let
        rho_rows = (O*R + 2) * 2^-52 * (max |Rbar| + gamma * m * max |x|),     m = max_{s,a} sum_{o,r} RTO[s,a,o,r]:
    an entry of a row of H V is Rbar + ((G_0 + G_1) + ...), G_o = gamma * sum_r RTO * x; a product term passes through at most R + O + 1 <=
    O*R + 2 roundings (the product, R - 1 additions, gamma, O - 1 additions, Rbar), each of relative size <= 2^-53, and the terms' magnitudes
    sum to at most max |Rbar| + gamma * m * max |x|; 2^-52 per rounding absorbs the second-order terms.  Pruning removes only rows that kept
    rows beat everywhere, so |V'(b) - (H V)(b)| <= rho_rows at every belief.  u_i itself is max_s (y_i - sum_q lambda_q x_{J_q})[s] computed
    with at most 64 fused multiply-adds and one subtraction, with lambda summing to 1 up to the rounding of its normalisation:
        rho_u = (64 + 2) * 2^-52 * (max |y| + max |x|)
    covers both.  With rho = rho_rows + rho_u and
        e = max(0, max_i u_i) + rho
    we have H V <= V + e at every belief.  H is monotone and H(V + c) <= H V + gamma' c for constants c >= 0, gamma' = gamma * max(1, m)
    (`certificate_contraction`), so H^{k+1} V <= H^k V + gamma'^k e and
        V* <= H V + gamma' e / (1 - gamma') <= V' + shift,     shift = gamma' e / (1 - gamma') + rho_rows
    at every belief (the last term: V' is H V as computed).  Where `certificate_contraction` raises, no shift is reported.  In exact
    arithmetic V' <= V* when the start is <= V* (H is monotone and V* = H V*); for a lower end that holds under rounding, extract a controller:
    `PolicyGraph.from_value_function(model, V').evaluate(gamma)`.

    Parameters
    ----------
    gamma : discount factor in (0, 1)
    eps : tolerance of the residual LP: a row's bounds stop when u_i - m*_i <= eps * max(1, max |V'|)
    max_candidates : the largest cross sum an epoch may build (rows); a larger one stops the solve with the last completed epoch
    """

    def __init__(self, gamma: float = 0.95, eps: float = 1e-10, max_candidates: int = 4_000_000):
        if not 0.0 < gamma < 1.0:
            raise ValueError('gamma must lie in (0, 1)')
        if not eps >= 0.0:
            raise ValueError('eps must be >= 0')
        self.gamma, self.eps, self.max_candidates = float(gamma), float(eps), int(max_candidates)

    # ---- one prune: pointwise dominance, then LP dominance --------------------------------------------------------------------------
    def _prune(self, dev, rows: torch.Tensor, tuples: np.ndarray, acc: dict) -> tuple:
        t0 = time.perf_counter()
        witness = dev.dominating_row(rows)
        keep = np.flatnonzero(witness.cpu().numpy() < 0)
        acc['dropped_pointwise'] += rows.shape[0] - keep.shape[0]
        if keep.shape[0] != rows.shape[0]:
            rows, tuples = rows[torch.as_tensor(keep, device=rows.device)], tuples[keep]
        t1 = time.perf_counter()
        acc['seconds']['pointwise'] += t1 - t0
        lp_keep, _, counts = dev.prune_lp(rows)
        total = acc['prune_lp_stats']
        for k, v in dev.prune_lp_stats().items():
            total[k] = max(total.get(k, 0), v) if k == 'max_competitors' else total.get(k, 0) + v
        acc['dropped_lp'] += int(counts[2])
        acc['undecided'] += int(counts[3])
        keep = np.flatnonzero(lp_keep.cpu().numpy() != 0)
        if keep.shape[0] != rows.shape[0]:
            rows, tuples = rows[torch.as_tensor(keep, device=rows.device)], tuples[keep]
        acc['seconds']['lp'] += time.perf_counter() - t1
        return rows.contiguous(), tuples

    def _cross_sum(self, dev, x, g, a: int, acc: dict) -> torch.Tensor:
        n = (1 if x is None else x.shape[0]) * g.shape[0]
        if n > self.max_candidates:
            raise _Candidates()
        t0 = time.perf_counter()
        out = dev.ip_cross_sum(x, g, a)
        torch.cuda.synchronize(dev.device)
        acc['seconds']['cross_sum'] += time.perf_counter() - t0
        return out

    def _epoch(self, model: Model, X: torch.Tensor) -> tuple:
        """V' = H V from the rows X: (rows, tuples [n, 1 + O], stats dict).  Raises _Candidates when a cross sum exceeds max_candidates."""
        dev = model.device
        A, O = model.action_count, model.observation_count
        acc = dict(fold_candidates=[], dropped_pointwise=0, dropped_lp=0, undecided=0, prune_lp_stats={},
                   seconds=dict(project=0.0, cross_sum=0.0, pointwise=0.0, lp=0.0, residual=0.0))
        parts, part_tuples = [], []
        ids = np.arange(X.shape[0], dtype=np.int64)
        for a in range(A):
            t0 = time.perf_counter()
            G = dev.ip_project(X, self.gamma, a)
            torch.cuda.synchronize(dev.device)
            acc['seconds']['project'] += time.perf_counter() - t0
            proj = [self._prune(dev, G[o].contiguous(), ids, acc) for o in range(O)]
            largest = 0
            if O == 1:
                largest = proj[0][0].shape[0]
                rows, tup = self._prune(dev, self._cross_sum(dev, None, proj[0][0], a, acc), proj[0][1][:, None], acc)
            else:
                rows, tup = proj[0][0], proj[0][1][:, None]
                for o in range(1, O):
                    g, gid = proj[o]
                    largest = max(largest, rows.shape[0] * g.shape[0])
                    cand = self._cross_sum(dev, rows, g, a if o == O - 1 else -1, acc)
                    rows, tup = self._prune(dev, cand, tuple_product(tup, gid), acc)
            acc['fold_candidates'].append(int(largest))
            parts.append(rows)
            part_tuples.append(np.concatenate([np.full((tup.shape[0], 1), a, dtype=np.int64), tup], axis=1))
        union = torch.cat(parts).contiguous()
        acc['union_candidates'] = int(union.shape[0])
        rows, tuples = self._prune(dev, union, np.concatenate(part_tuples), acc)
        return rows, tuples, acc

    # ---- the solve ---------------------------------------------------------------------------------------------------------------------
    def solve(self, model: Model, horizon: int = 1000, initial_value_function: ValueFunction | None = None, target: float | None = None,
              time_limit: float | None = None, print_progress: bool = False) -> tuple:
        """
        Up to `horizon` epochs V <- H V from the start V_0: returns (ValueFunction, IncrementalPruningHistory).

        V_0 is `initial_value_function` (any finite rows, e.g. one zero row: then V_H is the exact H-step value) or, by default, the
        certified rows of the blind controller (`PolicyGraph.blind(model).evaluate(gamma)`), which lie below V* for rewards of either sign.
        The solve stops after the first epoch whose shift is <= `target` ('target'), after `horizon` epochs ('horizon'), once `time_limit`
        seconds have passed ('time'), or when an epoch would build a cross sum of more than `max_candidates` rows ('candidates': the last
        completed epoch and its certificate are returned).  The rows of the returned value function carry the actions of their tuples.
        """
        t_start = time.perf_counter()
        S, A, O, R = model.state_count, model.action_count, model.observation_count, model.reachable_state_count
        if initial_value_function is None:
            from .policy_graph import PolicyGraph
            try:
                X, _ = PolicyGraph.blind(model).evaluate(self.gamma)
            except ValueError as err:
                raise ValueError(f'the default start needs a certified blind controller ({err}): pass initial_value_function') from err
            x_actions = np.arange(A, dtype=np.int64)
        else:
            X = initial_value_function.alpha_vector_array
            x_actions = np.asarray(initial_value_function.actions, dtype=np.int64)
        if X.dim() != 2 or X.shape[0] == 0 or X.shape[1] != S or not bool(torch.isfinite(X).all()):
            raise ValueError(f'the start value function needs at least one row of {S} finite entries')
        dev = model.device
        X = X.to(device=dev.device, dtype=torch.float64).contiguous()
        try:
            gamma_c = certificate_contraction(model, self.gamma, 'incremental pruning')
        except ValueError:
            gamma_c = None
        rbar = np.asarray(model.expected_rewards_table, dtype=np.float64)
        rto_mass = float(np.max(np.asarray(model.reachable_transitional_observation_table, dtype=np.float64).sum(axis=(2, 3))))
        rbar_max = float(np.max(np.abs(rbar)))
        history = IncrementalPruningHistory(self.gamma, self.eps)
        V = ValueFunction(model, X, x_actions)
        for epoch in range(1, int(horizon) + 1):
            try:
                Y, tuples, acc = self._epoch(model, X)
            except _Candidates:
                history.stopped = 'candidates'
                break
            if Y.shape[0] == 0 or not bool(torch.isfinite(Y).all()):
                raise ValueError('the backed-up rows are not finite')
            t0 = time.perf_counter()
            y_max, x_max = float(Y.abs().max()), float(X.abs().max())
            res = dev.ip_residual_lp(Y, X, self.eps * max(1.0, y_max))
            max_u = float(res['u'].max())
            acc['seconds']['residual'] = time.perf_counter() - t0
            rho_rows, rho_u = rounding_allowance(O, R, rbar_max, self.gamma, rto_mass, x_max, y_max)
            e = max(0.0, max_u) + rho_rows + rho_u
            shift = None if gamma_c is None else gamma_c * e / (1.0 - gamma_c) + rho_rows
            history.epochs.append(dict(epoch=epoch, rows=int(Y.shape[0]), **acc, residual_stats=res['stats'], max_u=max_u, e=e, shift=shift,
                                       elapsed=time.perf_counter() - t_start))
            history.previous, history.tuples, history.e, history.shift = X, tuples, e, shift
            X = Y
            V = ValueFunction(model, Y, tuples[:, 0])
            if print_progress:
                log(f'IncrementalPruning: epoch {epoch}, {Y.shape[0]} rows, max u = {max_u:.3e}, shift = {shift}')
            if shift is not None and target is not None and shift <= target:
                history.stopped = 'target'
                break
            if time_limit is not None and time.perf_counter() - t_start >= time_limit:
                history.stopped = 'time'
                break
        else:
            history.stopped = 'horizon'
        history.seconds = time.perf_counter() - t_start
        return V, history
