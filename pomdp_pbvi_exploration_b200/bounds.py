"""
Certified upper bounds on V*, so that the optimality gap upper(b) - lower(b) of any solve can be measured.

    FIB_Solver    the Fast Informed Bound (Hauskrecht 2000): A vectors U_a with max_a U_a . b >= V*(b) at every belief, one
                  `pbvi_fib_sweep` launch per iteration and a residual certificate at the end
    UpperBound    min(FIB bound, sawtooth over stored (belief, value) pairs), tightened by point-based upper-bound backups over a
                  belief set (`pbvi_upper_backup`); `gap(value_function)` returns (lower, upper) at the start belief

The HSVI upper bound (`solver.BeliefValueMapping`) is a separate object and is not touched by anything here.
"""
from __future__ import annotations

from datetime import datetime
from typing import Union

import numpy as np
import torch

from .belief import Belief, BeliefSet
from .model import Model, log
from .solver import MDPSolverHistory
from .value_function import ValueFunction

CHUNK_BYTES = 2 << 30        # per pbvi_upper_backup call: successors (n*A*O*S doubles) and sawtooth terms (n*A*O*(n_ub+1)) each stay below


def certificate_contraction(model: Model, gamma: float, what: str) -> float:
    """gamma' = gamma * max(1, m) with m = max_{s,a} sum_{o,r} RTO[s,a,o,r]: the factor by which a constant shift of every row passes through
    one sweep at most.  The residual certificates (FIB_Solver: upper bound, PolicyGraph.evaluate: lower bound) need gamma' < 1;
    otherwise this raises ValueError."""
    rto = np.asarray(model.reachable_transitional_observation_table, dtype=np.float64)
    m = float(np.max(rto.sum(axis=(2, 3))))
    gamma_c = float(gamma) * max(1.0, m)
    if not gamma_c < 1.0:
        raise ValueError(f'gamma * max(1, max_(s,a) sum_(o,r) RTO) = {gamma_c} >= 1: the {what} certificate needs a contraction')
    return gamma_c


def belief_rows(model: Model, beliefs) -> torch.Tensor:
    """A BeliefSet, a Belief, or an array / tensor of one or more rows as a contiguous CUDA float64 [n,S] tensor; non-finite rows raise
    ValueError."""
    if isinstance(beliefs, BeliefSet):
        rows = beliefs.belief_array
    elif isinstance(beliefs, Belief):
        rows = beliefs.values[None, :]
    else:
        rows = beliefs if isinstance(beliefs, torch.Tensor) else torch.as_tensor(np.asarray(beliefs, dtype=np.float64))
        if rows.dim() == 1:
            rows = rows[None, :]
    rows = rows.to(device=model.device.device, dtype=torch.float64).contiguous()
    if rows.dim() != 2 or rows.shape[1] != model.state_count:
        raise ValueError(f'beliefs must be [n, {model.state_count}], got {tuple(rows.shape)}')
    if rows.shape[0] and not bool(torch.isfinite(rows).all()):
        raise ValueError('belief rows must be finite')
    return rows


class FIB_Solver:
    """
    Fast Informed Bound value iteration (Hauskrecht 2000) on the device:

        (H U)_a[s] = Rbar[s,a] + gamma * sum_o max_{a'} sum_r RTO[s,a,o,r] * U_{a'}[reach[s,a,r]]

    Start: all A rows equal max Rbar / (1 - gamma), or one sweep of a user-supplied value function (any row count) to A rows.
    Stop: max |U_new - U| < eps * gamma / (1 - gamma) (one scalar read back per sweep), or `horizon` sweeps.

    Certificate (sound whatever the start, the stopping point or the rounding of the iterates): one more sweep gives the residual
    d = max(H U - U); with m = max_{s,a} sum_{o,r} RTO[s,a,o,r] and gamma' = gamma * max(1, m) the returned rows are
    U + max(d, 0) / (1 - gamma').  A constant shift c of every row passes through H as gamma * m(s,a) * c <= gamma' * c, so the returned
    rows satisfy H U <= U row by row.  Pushing b. through the inner maximum gives max_a (H U)_a . b >= (H_belief U^)(b) for
    U^(b) = max_a U_a . b, hence U^ >= H_belief U^, and since H_belief is a gamma'-contraction that is monotone, U^ >= V* at every belief.
    gamma' >= 1 (a model whose RTO rows sum to more than 1) raises ValueError.  The history records d (`fib_residual`) and the applied
    shift (`fib_shift`).
    """

    def __init__(self, horizon: int = 10000, gamma: float = 0.99, eps: float = 0.001):
        self.horizon = horizon
        self.gamma = gamma
        self.eps = eps

    def solve(self, model: Model, initial_value_function: Union[ValueFunction, None] = None, print_progress: bool = True,
              history_tracking_level: int = 1):
        """Returns (ValueFunction with one row per action, byte-deduplicated; MDPSolverHistory)."""
        gamma = float(self.gamma)
        gamma_c = certificate_contraction(model, gamma, 'FIB')
        dev = model.device
        A, S = model.action_count, model.state_count
        if initial_value_function is None:
            top = float(np.max(model.expected_rewards_table)) / (1.0 - gamma)
            U = torch.full((A, S), top, dtype=torch.float64, device=dev.device)
            V0 = ValueFunction(model, U, model.actions)
        else:
            V0 = initial_value_function
            if len(V0) == 0 or not bool(torch.isfinite(V0.alpha_vector_array).all()):
                raise ValueError('the initial value function must have at least one row and finite entries')
            U = dev.fib_sweep(V0.alpha_vector_array, gamma)
        history = MDPSolverHistory(history_tracking_level, model, gamma, self.eps, V0)
        max_allowed_change = self.eps * (gamma / (1 - gamma))
        for _ in range(self.horizon):
            start = datetime.now()
            U_new, stats = dev.fib_sweep(U, gamma, want_stats=True)
            max_change = float(stats[1])                                   # one scalar D2H per sweep = the convergence test
            U = U_new
            history.add((datetime.now() - start).total_seconds(), max_change,
                        ValueFunction(model, U.clone(), model.actions) if history_tracking_level >= 2 else None)
            if max_change < max_allowed_change:
                break
        _, stats = dev.fib_sweep(U, gamma, want_stats=True)
        residual = float(stats[0])
        if residual != residual:
            raise ValueError('the FIB iterates are not finite')
        shift = max(residual, 0.0) / (1.0 - gamma_c)
        if shift > 0.0:
            U = U + shift
        history.fib_residual, history.fib_shift = residual, shift
        if print_progress:
            log(f'FIB: {len(history.iteration_times)} sweeps, residual max(HU - U) = {residual:.3e}, certificate shift {shift:.3e}')
        return ValueFunction(model, U, model.actions), history


class UpperBound:
    """
    Upper bound on V*:  upper(b) = min( max_a F_a . b , sawtooth(b) )  for FIB rows F (`FIB_Solver`, or any rows with max_a F_a . b >= V*)
    and the sawtooth over stored (belief, value) pairs with corner values max_a F_a[s].

    `improve(belief_set)` runs point-based upper-bound backups u(b) = max_a [ b.Rbar_a + gamma sum_o P(o|b,a) upper(b^{ao}) ] over the set
    in reverse order, one chunk per `pbvi_upper_backup` call (every chunk sees the store as the previous chunk left it), and stores u(b)
    for each belief where u(b) < upper(b) -- a new pair, or a lower value for a stored belief (identity: the 128-bit row key).  Backups of
    an upper bound of V* are upper bounds of V*, and the sawtooth of upper bounds is one, so the bound stays sound; stored values only
    ever decrease.  The store is this object's own; HSVI's `BeliefValueMapping` is a different object.
    """

    def __init__(self, model: Model, fib: ValueFunction, gamma: float):
        self.model = model
        self.gamma = float(gamma)
        self.fib = fib
        F = fib.alpha_vector_array.contiguous()
        if F.shape[0] == 0 or not bool(torch.isfinite(F).all()):
            raise ValueError('the FIB rows must be finite and at least one')
        self._F = F
        self.corner_values = torch.max(F, dim=0).values.contiguous()
        self._chunk_bytes = CHUNK_BYTES
        self._n = 0
        self._cap = 0
        self._rows = self._vals = self._idx = self._val = self._count = self._dot = None
        self._index = {}                 # 128-bit row key -> position in the store

    # ---- store ------------------------------------------------------------------------------------------------------------
    def __len__(self) -> int:
        return self._n

    @property
    def belief_array(self) -> torch.Tensor:
        """[n,S] stored beliefs (CUDA float64)."""
        return self._rows[:self._n] if self._n else torch.empty((0, self.model.state_count), dtype=torch.float64, device=self._F.device)

    @property
    def value_array(self) -> torch.Tensor:
        """[n] stored values (CUDA float64)."""
        return self._vals[:self._n] if self._n else torch.empty((0,), dtype=torch.float64, device=self._F.device)

    def _reserve(self, n: int) -> None:
        if n <= self._cap:
            return
        dev, S = self._F.device, self.model.state_count
        cap = max(64, 2 * n)

        def grown(old, shape, dtype):
            t = torch.empty(shape, dtype=dtype, device=dev)
            if old is not None and self._n:
                t[:self._n] = old[:self._n]
            return t
        self._rows = grown(self._rows, (cap, S), torch.float64)
        self._vals = grown(self._vals, (cap,), torch.float64)
        self._idx = grown(self._idx, (cap, S), torch.int32)
        self._val = grown(self._val, (cap, S), torch.float64)
        self._count = grown(self._count, (cap,), torch.int32)
        self._dot = grown(self._dot, (cap,), torch.float64)
        self._cap = cap

    def _rows_of(self, beliefs) -> torch.Tensor:
        return belief_rows(self.model, beliefs)

    def _lists(self):
        n = self._n
        if n == 0:
            return None, None, None, None, None, 0
        return self._idx, self._val, self._count, self._dot, self._vals, n

    # ---- queries ----------------------------------------------------------------------------------------------------------
    def evaluate(self, belief_set) -> torch.Tensor:
        """upper(b) = min(max_a F_a . b, sawtooth(b)) for every row: CUDA float64 [n]."""
        dev = self.model.device
        rows = self._rows_of(belief_set)
        if rows.shape[0] == 0:
            return torch.empty((0,), dtype=torch.float64, device=rows.device)
        fib = dev.max_values(rows, self._F)[0]
        idx, val, count, dot, vals, n_ub = self._lists()
        saw = dev.sawtooth_lists(self.corner_values, idx, val, count, dot, vals, n_ub, rows)
        return torch.minimum(fib, saw)

    def gap(self, value_function: ValueFunction, belief=None) -> tuple:
        """(lower, upper) at `belief` (default: the model's start belief): lower = max_v alpha_v . b, upper = `evaluate`."""
        b = self.model.start_probabilities if belief is None else belief
        rows = self._rows_of(b)[:1]
        lower = float(self.model.device.max_values(rows, value_function.alpha_vector_array)[0][0])
        return lower, float(self.evaluate(rows)[0])

    # ---- point-based backups ----------------------------------------------------------------------------------------------
    def _chunk(self, n_left: int) -> int:
        m = self.model
        nZ = m.action_count * m.observation_count
        per_succ = nZ * m.state_count * 8
        per_saw = nZ * (self._n + 1) * 8
        return max(1, min(n_left, self._chunk_bytes // per_succ, self._chunk_bytes // per_saw))

    def improve(self, belief_set, passes: int = 1) -> tuple:
        """
        `passes` sweeps of upper-bound backups over the set, last belief first.  Returns (n_decreased, largest_decrease): how many
        backups lowered the bound at their belief (stored as a new pair, or a stored value lowered), and the largest upper(b) - u(b).
        """
        dev = self.model.device
        rows = self._rows_of(belief_set).flip(0).contiguous()
        n = rows.shape[0]
        n_dec, largest = 0, 0.0
        if n == 0:
            return n_dec, largest
        keys = dev.row_hash(rows).cpu().numpy()
        for _ in range(passes):
            i0 = 0
            while i0 < n:
                nc = self._chunk(n - i0)
                idx, val, count, dot, vals, n_ub = self._lists()
                u, cur = dev.upper_backup(rows[i0:i0 + nc], self._F, self.gamma, self.corner_values, idx, val, count, dot, vals, n_ub)
                u_h, cur_h = u.cpu().numpy(), cur.cpu().numpy()
                hit = np.flatnonzero(u_h < cur_h)
                if hit.size:
                    n_dec += int(hit.size)
                    largest = max(largest, float(np.max(cur_h[hit] - u_h[hit])))
                    self._store(rows, keys, i0, hit, u_h)
                i0 += nc
        return n_dec, largest

    def _store(self, rows: torch.Tensor, keys: np.ndarray, i0: int, hit: np.ndarray, u_h: np.ndarray) -> None:
        """Stores u for the chunk rows `hit` (offsets from i0): new pairs are appended (support lists built for them), stored beliefs
        get min(stored, u)."""
        new_rows, new_vals, low_pos, low_vals = [], [], [], []
        for j in hit.tolist():
            key = (int(keys[i0 + j, 0]), int(keys[i0 + j, 1]))
            pos = self._index.get(key)
            if pos is None:
                self._index[key] = self._n + len(new_rows)
                new_rows.append(i0 + j)
                new_vals.append(float(u_h[j]))
            elif pos >= self._n:                                   # twice in this chunk: same row, same u
                continue
            else:
                low_pos.append(pos)
                low_vals.append(float(u_h[j]))
        dev_t = self._F.device
        if low_pos:
            p = torch.as_tensor(low_pos, dtype=torch.int64, device=dev_t)
            self._vals[p] = torch.minimum(self._vals[p], torch.as_tensor(low_vals, dtype=torch.float64, device=dev_t))
        if new_rows:
            lo, k = self._n, len(new_rows)
            self._reserve(lo + k)
            self._rows[lo:lo + k] = rows[torch.as_tensor(new_rows, dtype=torch.int64, device=dev_t)]
            self._vals[lo:lo + k] = torch.as_tensor(new_vals, dtype=torch.float64, device=dev_t)
            self.model.device.support_lists(self._rows[lo:lo + k], self.corner_values, self._idx[lo:lo + k], self._val[lo:lo + k],
                                            self._count[lo:lo + k], self._dot[lo:lo + k])
            self._n = lo + k
