"""
ctypes binding of libpbvi_b200.so (C ABI in include/pbvi_b200.h) -- the only compute path of the package.

PyTorch is used for device memory, streams and (in `parallel.py`) torch.distributed; every kernel is the
library's.  There is no CPU fallback: importing this module without the built library, or creating a
`DeviceModel` without a CUDA device, raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, byref, c_char_p, c_double, c_int, c_int32, c_int64, c_uint64, c_void_p

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('PBVI_B200_LIB', os.path.join(_HERE, 'libpbvi_b200.so'))     # override: A/B builds of the same engine

PBVI_OK, PBVI_ERR_BAD_ARG, PBVI_ERR_CUDA, PBVI_ERR_OOM, PBVI_ERR_UNSUPPORTED, PBVI_ERR_NCCL = 0, -1, -2, -3, -4, -5

# name -> argtypes; every function returns int except pbvi_last_error.  Kept in one table so that the CPU test-suite can
# check the library exports exactly what include/pbvi_b200.h declares.
_P = c_void_p
SIGNATURES = {
    'pbvi_version': [],
    'pbvi_model_create': [c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_int, POINTER(c_void_p)],
    'pbvi_model_destroy': [_P],
    'pbvi_model_dims': [_P, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int)],
    'pbvi_backup_select': [_P, _P, c_int, _P, c_int, c_double, _P, _P, _P, _P],
    'pbvi_backup_assemble': [_P, _P, c_int, c_double, _P, _P, c_int, _P, _P, _P],
    'pbvi_controller_sweep': [_P, _P, c_int, c_double, _P, _P, _P, _P, _P],
    'pbvi_controller_evaluate': [_P, _P, c_int, c_double, _P, _P, c_double, c_int, _P, _P, POINTER(c_int), _P],
    'pbvi_controller_outcomes': [_P, c_int, _P, _P, _P, _P, c_double, c_int, _P, _P, c_int, _P, _P, _P, _P, _P],
    'pbvi_controller_evaluate_mixed': [_P, _P, c_int, c_double, _P, _P, c_int, _P, _P, _P, c_double, c_int, _P, _P, POINTER(c_int), _P],
    'pbvi_controller_outcomes_mixed': [_P, c_int, _P, _P, c_int, _P, _P, _P, _P, _P, c_double, c_int, _P, _P, c_int, _P, _P, _P, _P, _P],
    'pbvi_backup': [_P, _P, c_int, _P, c_int, c_double, _P, _P, _P, _P, _P],
    'pbvi_backup_host': [_P, _P, c_int, _P, c_int, c_double, _P, _P, _P],
    'pbvi_backup_host_unique': [_P, _P, c_int, _P, c_int, c_double, _P, c_int, _P, POINTER(c_int), _P],
    'pbvi_backup_small_eligible': [_P, c_int, c_int],
    'pbvi_backup_small': [_P, _P, c_int, _P, c_int, c_double, _P, _P, _P, POINTER(c_int), _P],
    'pbvi_max_values': [_P, _P, c_int, _P, c_int, _P, _P, _P],
    'pbvi_belief_update': [_P, _P, _P, _P, c_int, c_int, _P, _P, _P],
    'pbvi_belief_trajectory': [_P, _P, _P, _P, _P, c_int, _P, _P],
    'pbvi_perseus_walk': [_P, _P, _P, _P, c_int, _P, _P, _P],
    'pbvi_belief_successors': [_P, _P, c_int, c_int, _P, _P, _P],
    'pbvi_observation_probabilities': [_P, _P, c_int, _P, _P],
    'pbvi_row_hash': [_P, _P, c_int, c_int, _P, _P],
    'pbvi_rows_equal': [_P, _P, _P, _P, _P, c_int, c_int, _P, _P],
    'pbvi_group_keys': [_P, _P, c_int, c_int, _P, _P, _P, _P, POINTER(c_int), _P],
    'pbvi_group_record_blocks': [_P, _P, c_int, c_int, c_int, _P, _P, POINTER(c_int), POINTER(c_int), _P],
    'pbvi_confirm_groups': [_P, _P, c_int, c_int, _P, _P, POINTER(c_int), _P],
    'pbvi_pack_rows_host': [_P, c_int, c_int, _P, _P, _P, POINTER(c_int64)],
    'pbvi_pack_slabs_host': [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int64, _P],
    'pbvi_unpack_rows': [_P, _P, _P, _P, c_int, c_int, c_int, c_int64, _P, _P],
    'pbvi_vi_sweep': [_P, _P, c_double, _P, _P, _P],
    'pbvi_fib_sweep': [_P, _P, c_int, c_double, _P, _P, _P],
    'pbvi_upper_backup': [_P, _P, c_int, _P, c_int, c_double, _P, _P, _P, _P, _P, _P, c_int, _P, _P, _P, _P],
    'pbvi_prune_dominated': [_P, _P, c_int, _P, _P],
    'pbvi_first_dominating_row': [_P, _P, c_int, _P, c_int, _P, _P],
    'pbvi_dominating_row': [_P, _P, c_int, _P, _P],
    'pbvi_prune_lp': [_P, _P, c_int, _P, _P, _P, _P],
    'pbvi_prune_lp_certificates': [_P, _P, c_int, _P, _P, _P, _P, _P, _P],
    'pbvi_prune_lp_stats': [_P, _P],
    'pbvi_bpi_lp': [_P, _P, c_int, c_int, c_double, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    'pbvi_ip_project': [_P, _P, c_int, c_double, c_int, _P, _P],
    'pbvi_ip_cross_sum': [_P, _P, c_int, _P, c_int, c_int, _P, _P],
    'pbvi_ip_residual_lp': [_P, _P, c_int, _P, c_int, c_double, _P, _P, _P, _P, _P, _P, _P],
    'pbvi_sawtooth': [_P, _P, _P, _P, c_int, _P, c_int, _P, _P],
    'pbvi_support_lists': [_P, _P, c_int, _P, _P, _P, _P, _P, _P],
    'pbvi_sawtooth_lists': [_P, _P, _P, _P, _P, _P, _P, c_int, _P, c_int, _P, _P],
    'pbvi_sawtooth_witness': [_P, _P, _P, _P, _P, _P, _P, c_int, _P, _P, _P, _P],
    'pbvi_hsvi_level': [_P, _P, _P, c_int, c_double, _P, _P, _P, _P, _P, _P, c_int, _P, _P, c_int, c_int, c_double, c_int, _P, _P, _P, _P, _P],
    'pbvi_gap_trial_step': [_P, _P, c_int, _P, c_int, _P, c_int, c_double, _P, _P, _P, _P, _P, _P, c_int, c_double, _P, _P, _P, _P, _P, _P],
    'pbvi_min_l2_distance': [_P, _P, c_int, _P, c_int, _P, _P],
    'pbvi_ger_scores': [_P, _P, _P, _P, c_int, c_double, c_double, _P, _P],
    'pbvi_comm_unique_id': [_P],
    'pbvi_comm_init': [_P, _P, c_int, c_int, POINTER(c_void_p)],
    'pbvi_comm_destroy': [_P],
    'pbvi_comm_rank': [_P, POINTER(c_int), POINTER(c_int)],
    'pbvi_allgather_tuples': [_P, _P, c_int, c_int, _P, _P],
    'pbvi_allgather_rows': [_P, _P, c_int, c_int, _P, _P],
    'pbvi_allreduce_max': [_P, _P, c_int, _P],
    'pbvi_broadcast_rows': [_P, _P, ctypes.c_size_t, c_int, _P],
    'pbvi_last_stats': [_P, POINTER(c_double), POINTER(c_double), POINTER(c_int)],
    'pbvi_last_launches': [_P],
    'pbvi_set_option': [_P, c_char_p, c_int],
    'pbvi_set_profiling': [_P, c_int],
    'pbvi_last_score_ms': [_P, POINTER(ctypes.c_float)],
}

_lib = None


def load_library() -> ctypes.CDLL:
    """Loads the engine.  Raises (never falls back) when it has not been built: run `python -m pomdp_pbvi_exploration_b200.build`."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} is missing: build it with `python -m pomdp_pbvi_exploration_b200.build` '
                           '(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = c_int
    lib.pbvi_last_error.argtypes = []
    lib.pbvi_last_error.restype = c_char_p
    _lib = lib
    return lib


class PBVIError(RuntimeError):
    pass


def _check(rc: int) -> None:
    if rc == PBVI_OK:
        return
    msg = load_library().pbvi_last_error().decode(errors='replace')
    if rc == PBVI_ERR_OOM:
        raise MemoryError(msg)          # the solve loop's `except MemoryError` keeps working (reference src/pomdp.py:2399)
    if rc == PBVI_ERR_BAD_ARG:
        raise ValueError(msg)
    raise PBVIError(f'libpbvi_b200 error {rc}: {msg}')


def _ptr(t) -> int:
    if t is None:
        return None
    return t.data_ptr()


def _f64(t: torch.Tensor, device) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.ascontiguousarray(t, dtype=np.float64))
    return t.to(device=device, dtype=torch.float64).contiguous()


def _i32(t, device) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.ascontiguousarray(t))
    return t.to(device=device, dtype=torch.int32).contiguous()


class DeviceModel:
    """
    Device-resident model tables + scratch (one `pbvi_model` handle).  Inputs are the reference's host tensors:
    reachable_states [S,A,R] int, reachable_probabilities [S,A,R], RTO [S,A,O,R], expected_rewards_table [S,A]
    (reference Model.gpu_model, src/mdp.py:533-560).  All methods take / return CUDA float64 / int32 torch tensors on
    `self.device` and enqueue on the current torch stream.
    """

    def __init__(self, reach: np.ndarray, probs: np.ndarray | None, rto: np.ndarray, rbar: np.ndarray, device: int | None = None):
        self._h = None
        self.launch_count = 0           # kernels launched through this handle since creation (bench.py: gpu_launches)
        self._lib = load_library()
        if not torch.cuda.is_available():
            raise RuntimeError('no CUDA device: the PBVI B200 engine has no CPU path')
        if device is None:
            device = torch.cuda.current_device()
        S, A, R = reach.shape
        O = rto.shape[2]
        assert rto.shape == (S, A, O, R) and rbar.shape == (S, A)
        reach64 = np.ascontiguousarray(reach, dtype=np.int64)
        rto64 = np.ascontiguousarray(rto, dtype=np.float64)
        rbar64 = np.ascontiguousarray(rbar, dtype=np.float64)
        probs64 = None if probs is None else np.ascontiguousarray(probs, dtype=np.float64)
        h = c_void_p()
        _check(self._lib.pbvi_model_create(S, A, O, R, reach64.ctypes.data, None if probs64 is None else probs64.ctypes.data,
                                           rto64.ctypes.data, rbar64.ctypes.data, int(device), byref(h)))
        self._h = h
        self.S, self.A, self.O, self.R = S, A, O, R
        self.device = torch.device('cuda', int(device))

    def _call(self, rc: int) -> None:
        _check(rc)
        self.launch_count += self._lib.pbvi_last_launches(self._h)

    def close(self) -> None:
        if self._h is not None:
            self._lib.pbvi_model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------
    @property
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _beliefs(self, beliefs) -> torch.Tensor:
        b = _f64(beliefs, self.device)
        if b.dim() == 1:
            b = b[None, :]
        assert b.dim() == 2 and b.shape[1] == self.S, f'beliefs must be [n, {self.S}], got {tuple(b.shape)}'
        return b

    def backup_select(self, beliefs, alphas, gamma: float, want_value: bool = True):
        """v*[b,a,o], value[b,a], a*[b] (reference src/pomdp.py:1485-1505)."""
        b, al = self._beliefs(beliefs), self._beliefs(alphas)
        nB, nV = b.shape[0], al.shape[0]
        vstar = torch.empty((nB, self.A, self.O), dtype=torch.int32, device=self.device)
        value = torch.empty((nB, self.A), dtype=torch.float64, device=self.device) if want_value else None
        astar = torch.empty((nB,), dtype=torch.int32, device=self.device)
        self._call(self._lib.pbvi_backup_select(self._h, _ptr(b), nB, _ptr(al), nV, float(gamma), _ptr(vstar), _ptr(value), _ptr(astar),
                                            self._stream))
        return vstar, value, astar

    def backup_assemble(self, alphas, gamma: float, actions, vsel, with_hash: bool = False):
        """alpha_a rows for (action, v*[O]) tuples (reference src/pomdp.py:1497-1506); `with_hash` also returns their 128-bit
        row keys (int64 [n,2], equal to `row_hash(rows)`) computed in the same pass."""
        al = self._beliefs(alphas)
        act, vs = _i32(actions, self.device), _i32(vsel, self.device)
        n = act.shape[0]
        assert vs.shape == (n, self.O)
        out = torch.empty((n, self.S), dtype=torch.float64, device=self.device)
        keys = torch.empty((n, 2), dtype=torch.int64, device=self.device) if with_hash else None
        self._call(self._lib.pbvi_backup_assemble(self._h, _ptr(al), al.shape[0], float(gamma), _ptr(act), _ptr(vs), n, _ptr(out),
                                                  _ptr(keys), self._stream))
        return (out, keys) if with_hash else out

    def controller_sweep(self, rows, gamma: float, actions, succ, want_stats: bool = False):
        """One evaluation sweep of a finite-state controller (`pbvi_controller_sweep`): n rows [n,S] from the n node rows `rows`, node i
        playing actions[i] and moving to succ[i][o]; with `want_stats` also the device triple {max(out - rows), max(rows - out),
        max |out - rows|} [3] computed by the same launch."""
        W = self._beliefs(rows)
        act, sc = _i32(actions, self.device), _i32(succ, self.device)
        n = W.shape[0]
        assert act.shape == (n,) and sc.shape == (n, self.O)
        out = torch.empty((n, self.S), dtype=torch.float64, device=self.device)
        stats = torch.empty((3,), dtype=torch.float64, device=self.device) if want_stats else None
        self._call(self._lib.pbvi_controller_sweep(self._h, _ptr(W), n, float(gamma), _ptr(act), _ptr(sc), _ptr(out), _ptr(stats), self._stream))
        return (out, stats) if want_stats else out

    def controller_evaluate(self, rows, gamma: float, actions, succ, tol: float, max_sweeps: int):
        """Up to `max_sweeps` controller sweeps in one persistent launch (`pbvi_controller_evaluate`), stopping after the first whose
        max |out - in| is below `tol` or NaN: returns (last iterate [n,S], per-sweep max |out - in| [k] CUDA float64, k).  Synchronises."""
        W = self._beliefs(rows)
        act, sc = _i32(actions, self.device), _i32(succ, self.device)
        n = W.shape[0]
        assert act.shape == (n,) and sc.shape == (n, self.O)
        out = torch.empty((n, self.S), dtype=torch.float64, device=self.device)
        changes = torch.empty((max(int(max_sweeps), 1),), dtype=torch.float64, device=self.device)
        k = c_int(0)
        self._call(self._lib.pbvi_controller_evaluate(self._h, _ptr(W), n, float(gamma), _ptr(act), _ptr(sc), float(tol), int(max_sweeps),
                                                      _ptr(out), _ptr(changes), byref(k), self._stream))
        return out, changes[:k.value], k.value

    def controller_outcomes(self, actions, succ, end_state, end_action, gamma: float, steps: int, queries, query_nodes):
        """`steps` sweeps of the outcome recursions of a controller whose runs stop at end states (`pbvi_controller_outcomes`, one
        persistent launch): returns (success, steps, return) rows [n,S] and the series [steps, q, 3] of b_j . {P, M, G}_k(query_nodes[j])
        after every sweep, CUDA float64.  `end_state` [S] / `end_action` [A] are flags (non-zero: ends).  Synchronises."""
        act, sc = _i32(actions, self.device), _i32(succ, self.device)
        n = act.shape[0]
        assert sc.shape == (n, self.O)
        es = torch.as_tensor(np.asarray(end_state) != 0, device=self.device).to(torch.uint8).contiguous()
        ea = torch.as_tensor(np.asarray(end_action) != 0, device=self.device).to(torch.uint8).contiguous()
        assert es.shape == (self.S,) and ea.shape == (self.A,)
        b = self._beliefs(queries)
        qn = _i32(query_nodes, self.device).reshape(-1)
        q = b.shape[0]
        assert qn.shape == (q,)
        P, M, G = (torch.empty((n, self.S), dtype=torch.float64, device=self.device) for _ in range(3))
        series = torch.empty((int(steps), q, 3), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_controller_outcomes(self._h, n, _ptr(act), _ptr(sc), _ptr(es), _ptr(ea), float(gamma), int(steps), _ptr(b),
                                                      _ptr(qn), q, _ptr(P), _ptr(M), _ptr(G), _ptr(series), self._stream))
        return P, M, G, series

    def _mixtures(self, mixtures):
        off, nodes, w = mixtures
        off, nodes, w = _i32(off, self.device).reshape(-1), _i32(nodes, self.device).reshape(-1), _f64(w, self.device).reshape(-1)
        assert off.shape[0] >= 1 and nodes.shape == w.shape
        return off.shape[0] - 1, off, nodes, w

    def controller_evaluate_mixed(self, rows, gamma: float, actions, succ, mixtures, tol: float, max_sweeps: int):
        """`controller_evaluate` of a controller with mixtures (`pbvi_controller_evaluate_mixed`): `mixtures` = (offsets [M+1], member
        nodes [nnz], weights [nnz]); a successor entry v >= n means mixture v - n.  Returns (last iterate [n,S], per-sweep max |out - in|
        over the n node rows [k] CUDA float64, k).  Synchronises."""
        W = self._beliefs(rows)
        act, sc = _i32(actions, self.device), _i32(succ, self.device)
        n = W.shape[0]
        assert act.shape == (n,) and sc.shape == (n, self.O)
        M, off, nodes, w = self._mixtures(mixtures)
        out = torch.empty((n, self.S), dtype=torch.float64, device=self.device)
        changes = torch.empty((max(int(max_sweeps), 1),), dtype=torch.float64, device=self.device)
        k = c_int(0)
        self._call(self._lib.pbvi_controller_evaluate_mixed(self._h, _ptr(W), n, float(gamma), _ptr(act), _ptr(sc), M, _ptr(off), _ptr(nodes),
                                                            _ptr(w), float(tol), int(max_sweeps), _ptr(out), _ptr(changes), byref(k),
                                                            self._stream))
        return out, changes[:k.value], k.value

    def controller_outcomes_mixed(self, actions, succ, mixtures, end_state, end_action, gamma: float, steps: int, queries, query_nodes):
        """`controller_outcomes` of a controller with mixtures (`pbvi_controller_outcomes_mixed`; `mixtures` as for
        `controller_evaluate_mixed`).  Synchronises."""
        act, sc = _i32(actions, self.device), _i32(succ, self.device)
        n = act.shape[0]
        assert sc.shape == (n, self.O)
        M, off, nodes, w = self._mixtures(mixtures)
        es = torch.as_tensor(np.asarray(end_state) != 0, device=self.device).to(torch.uint8).contiguous()
        ea = torch.as_tensor(np.asarray(end_action) != 0, device=self.device).to(torch.uint8).contiguous()
        assert es.shape == (self.S,) and ea.shape == (self.A,)
        b = self._beliefs(queries)
        qn = _i32(query_nodes, self.device).reshape(-1)
        q = b.shape[0]
        assert qn.shape == (q,)
        P, Mr, G = (torch.empty((n, self.S), dtype=torch.float64, device=self.device) for _ in range(3))
        series = torch.empty((int(steps), q, 3), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_controller_outcomes_mixed(self._h, n, _ptr(act), _ptr(sc), M, _ptr(off), _ptr(nodes), _ptr(w), _ptr(es),
                                                            _ptr(ea), float(gamma), int(steps), _ptr(b), _ptr(qn), q, _ptr(P), _ptr(Mr), _ptr(G),
                                                            _ptr(series), self._stream))
        return P, Mr, G, series

    def first_dominating_row(self, new_rows, old_rows) -> torch.Tensor:
        """For every row of `old_rows`, the first row of `new_rows` that is >= it at every state, or -1 (`pbvi_first_dominating_row`):
        int32 [n_old] CUDA tensor."""
        Y, X = self._beliefs(new_rows), self._beliefs(old_rows)
        first = torch.empty((X.shape[0],), dtype=torch.int32, device=self.device)
        self._call(self._lib.pbvi_first_dominating_row(self._h, _ptr(Y), Y.shape[0], _ptr(X), X.shape[0], _ptr(first), self._stream))
        return first

    def dominating_row(self, rows) -> torch.Tensor:
        """For every row, the smallest other row that is >= it at every state and, when it comes later, > it somewhere, or -1
        (`pbvi_dominating_row`): int32 [n] CUDA tensor."""
        X = self._beliefs(rows)
        witness = torch.empty((X.shape[0],), dtype=torch.int32, device=self.device)
        self._call(self._lib.pbvi_dominating_row(self._h, _ptr(X), X.shape[0], _ptr(witness), self._stream))
        return witness

    def backup(self, beliefs, alphas, gamma: float):
        """select + assemble for every belief, no dedup: (alpha [nB,S], action [nB], v* [nB,A,O], value [nB,A])."""
        b, al = self._beliefs(beliefs), self._beliefs(alphas)
        nB, nV = b.shape[0], al.shape[0]
        out = torch.empty((nB, self.S), dtype=torch.float64, device=self.device)
        act = torch.empty((nB,), dtype=torch.int32, device=self.device)
        vstar = torch.empty((nB, self.A, self.O), dtype=torch.int32, device=self.device)
        value = torch.empty((nB, self.A), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_backup(self._h, _ptr(b), nB, _ptr(al), nV, float(gamma), _ptr(out), _ptr(act), _ptr(vstar), _ptr(value),
                                     self._stream))
        return out, act, vstar, value

    def backup_small_eligible(self, n_beliefs: int, n_alphas: int) -> bool:
        """Mirror of the library's size rule (`pbvi_backup_small_eligible`), kept on the host: this path is about microseconds."""
        S, nZ = self.S, self.A * self.O
        return (0 < n_beliefs <= 16384 and 0 < n_alphas <= 4096 and S <= 1024 and (1 + nZ) * S + self.A + nZ <= 5000 and
                n_beliefs * S <= 262144 and float(n_beliefs) * n_alphas * nZ * S <= 6e7)

    def backup_small(self, beliefs: torch.Tensor, alphas: torch.Tensor, gamma: float):
        """Whole backup of a small problem in one library call (see `pbvi_backup_small`): returns (rows [n,S] CUDA tensor,
        actions [n] int64, row keys [n,2] int64) of the deduplicated new value function."""
        def ready(t):
            return isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64 and t.dim() == 2 and t.is_contiguous()
        b = beliefs if ready(beliefs) else self._beliefs(beliefs)
        al = alphas if ready(alphas) else self._beliefs(alphas)
        nB = b.shape[0]
        out = torch.empty((nB, self.S), dtype=torch.float64, device=self.device)
        acts = np.empty((nB,), dtype=np.int32)
        keys = np.empty((nB, 2), dtype=np.int64)
        n = c_int()
        _check(self._lib.pbvi_backup_small(self._h, b.data_ptr(), nB, al.data_ptr(), al.shape[0], float(gamma), out.data_ptr(), acts.ctypes.data,
                                           keys.ctypes.data, byref(n), self._stream))
        self.launch_count += 2                                   # the fused kernel + the gather
        k = n.value
        return out[:k], acts[:k].astype(np.int64), keys[:k]

    def backup_host(self, beliefs: np.ndarray, alphas: np.ndarray, gamma: float, out_alpha: np.ndarray | None = None,
                    out_action: np.ndarray | None = None):
        """Host-buffer entry point (copies inside): returns (alpha [nB,S] float64, action [nB] int32) NumPy arrays."""
        b = np.ascontiguousarray(beliefs, dtype=np.float64)
        al = np.ascontiguousarray(alphas, dtype=np.float64)
        nB, nV = b.shape[0], al.shape[0]
        if out_alpha is None:
            out_alpha = np.empty((nB, self.S), dtype=np.float64)
        if out_action is None:
            out_action = np.empty((nB,), dtype=np.int32)
        self._call(self._lib.pbvi_backup_host(self._h, b.ctypes.data, nB, al.ctypes.data, nV, float(gamma), out_alpha.ctypes.data,
                                          out_action.ctypes.data, self._stream))
        return out_alpha, out_action

    def backup_host_unique(self, beliefs: np.ndarray, alphas: np.ndarray, gamma: float):
        """The reference's whole backup from host arrays in one library call (`pbvi_backup_host_unique`): (rows [n,S], actions [n]) of
        the de-duplicated new value function, rows in order of first occurrence."""
        b = np.ascontiguousarray(beliefs, dtype=np.float64)
        al = np.ascontiguousarray(alphas, dtype=np.float64)
        nB, nV = b.shape[0], al.shape[0]
        out_alpha = np.empty((nB, self.S), dtype=np.float64)
        out_action = np.empty((nB,), dtype=np.int32)
        n = c_int()
        self._call(self._lib.pbvi_backup_host_unique(self._h, b.ctypes.data, nB, al.ctypes.data, nV, float(gamma), out_alpha.ctypes.data, nB,
                                                 out_action.ctypes.data, byref(n), self._stream))
        return out_alpha[:n.value], out_action[:n.value]

    def max_values(self, beliefs, alphas):
        """(max_v b.alpha_v, first argmax) -- reference src/pomdp.py:2165, 1639, 1735."""
        b, al = self._beliefs(beliefs), self._beliefs(alphas)
        nB = b.shape[0]
        mx = torch.empty((nB,), dtype=torch.float64, device=self.device)
        arg = torch.empty((nB,), dtype=torch.int32, device=self.device)
        self._call(self._lib.pbvi_max_values(self._h, _ptr(b), nB, _ptr(al), al.shape[0], _ptr(mx), _ptr(arg), self._stream))
        return mx, arg

    def belief_update(self, beliefs, actions, observations, normalise: bool = True):
        """Row-wise Belief.update (reference src/pomdp.py:382-421): returns (b' [n,S], mass [n])."""
        b = self._beliefs(beliefs)
        a, o = _i32(actions, self.device), _i32(observations, self.device)
        n = b.shape[0]
        assert a.shape == (n,) and o.shape == (n,)
        out = torch.empty((n, self.S), dtype=torch.float64, device=self.device)
        norm = torch.empty((n,), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_belief_update(self._h, _ptr(b), _ptr(a), _ptr(o), n, int(normalise), _ptr(out), _ptr(norm), self._stream))
        return out, norm

    def belief_trajectory(self, b0: torch.Tensor, actions, observations, resets=None) -> torch.Tensor:
        """Chain of updates from b0 following host (a, o) sequences; restarts from b0 after steps flagged in `resets`."""
        b = _f64(b0, self.device).reshape(-1)
        a = np.ascontiguousarray(actions, dtype=np.int32)
        o = np.ascontiguousarray(observations, dtype=np.int32)
        r = None if resets is None else np.ascontiguousarray(resets, dtype=np.uint8)
        n = a.shape[0]
        out = torch.empty((n, self.S), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_belief_trajectory(self._h, _ptr(b), a.ctypes.data, o.ctypes.data, None if r is None else r.ctypes.data, n,
                                                    _ptr(out), self._stream))
        return out

    def perseus_walk(self, b0: torch.Tensor, actions, uniforms, want_observations: bool = False):
        """Random walk in belief space from b0: host-drawn actions and uniforms, observations drawn on the device (see
        `pbvi_perseus_walk`).  Returns the n visited beliefs [n,S] (and the drawn observations [n] int32 when asked)."""
        b = _f64(b0, self.device).reshape(-1)
        a = np.ascontiguousarray(actions, dtype=np.int32)
        u = np.ascontiguousarray(uniforms, dtype=np.float64)
        n = a.shape[0]
        assert u.shape == (n,) and b.shape[0] == self.S
        out = torch.empty((n, self.S), dtype=torch.float64, device=self.device)
        obs = torch.empty((n,), dtype=torch.int32, device=self.device) if want_observations else None
        self._call(self._lib.pbvi_perseus_walk(self._h, _ptr(b), a.ctypes.data, u.ctypes.data, n, _ptr(out), _ptr(obs), self._stream))
        return (out, obs) if want_observations else out

    def belief_successors(self, beliefs, normalise: bool = True):
        """All (a,o) successors: (succ [n,A,O,S], mass [n,A,O]); NaN rows for impossible observations when normalised."""
        b = self._beliefs(beliefs)
        n = b.shape[0]
        out = torch.empty((n, self.A, self.O, self.S), dtype=torch.float64, device=self.device)
        norm = torch.empty((n, self.A, self.O), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_belief_successors(self._h, _ptr(b), n, int(normalise), _ptr(out), _ptr(norm), self._stream))
        return out, norm

    def observation_probabilities(self, beliefs) -> torch.Tensor:
        b = self._beliefs(beliefs)
        out = torch.empty((b.shape[0], self.A, self.O), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_observation_probabilities(self._h, _ptr(b), b.shape[0], _ptr(out), self._stream))
        return out

    def row_hash(self, rows: torch.Tensor) -> torch.Tensor:
        """128-bit hash of the raw bytes of each float64 row, as int64 [n,2]."""
        r = _f64(rows, self.device)
        out = torch.empty((r.shape[0], 2), dtype=torch.int64, device=self.device)
        self._call(self._lib.pbvi_row_hash(self._h, _ptr(r), r.shape[0], r.shape[1], _ptr(out), self._stream))
        return out

    def rows_equal(self, rows_a, ia, rows_b, ib) -> torch.Tensor:
        ra, rb = _f64(rows_a, self.device), _f64(rows_b, self.device)
        ia, ib = _i32(ia, self.device), _i32(ib, self.device)
        assert ra.shape[1] == rb.shape[1] and ia.shape == ib.shape
        flags = torch.empty((ia.shape[0],), dtype=torch.int32, device=self.device)
        self._call(self._lib.pbvi_rows_equal(self._h, _ptr(ra), _ptr(ia), _ptr(rb), _ptr(ib), ia.shape[0], ra.shape[1], _ptr(flags), self._stream))
        return flags

    def group_keys(self, keys: torch.Tensor, rank: torch.Tensor | None = None, want_inverse: bool = False):
        """
        Dict-insertion grouping of fixed-width integer keys on the device (reference src/mdp.py:668-669): `keys` is an int32
        [n,w] or int64 [n,w] CUDA tensor (viewed as 32-bit words).  Returns (first [g], last [g], inverse [n] | None) as int32
        CUDA tensors: groups in order of first occurrence, `last` = the record with the largest (rank, index).
        """
        k = keys.to(device=self.device).contiguous()
        n = k.shape[0]
        assert k.dim() == 2 and k.dtype in (torch.int32, torch.int64)
        words = k.shape[1] * (2 if k.dtype == torch.int64 else 1)
        first = torch.empty((n,), dtype=torch.int32, device=self.device)
        last = torch.empty((n,), dtype=torch.int32, device=self.device)
        inverse = torch.empty((n,), dtype=torch.int32, device=self.device) if want_inverse else None
        r = None if rank is None else _i32(rank, self.device)
        assert r is None or r.shape == (n,)
        count = c_int()
        self._call(self._lib.pbvi_group_keys(self._h, _ptr(k), n, words, _ptr(r), _ptr(first), _ptr(last), _ptr(inverse), byref(count),
                                             self._stream))
        return first[:count.value], last[:count.value], inverse

    def group_record_blocks(self, blocks: torch.Tensor, world: int, block_rows: int, words: int):
        """
        Merge of the all-gathered tuple blocks of a sharded backup (`parallel.exchange_tuples`): `blocks` is the int32 CUDA buffer
        [world * block_rows, words + 2]; returns (first_rows [g], last_rows [g], max_records) -- rows of the buffer holding the
        first record of every distinct key (ascending) and the record with the largest last position, and the largest record
        count any rank announced in its header.
        """
        assert blocks.dtype == torch.int32 and blocks.is_contiguous() and tuple(blocks.shape) == (world * block_rows, words + 2)
        n = world * block_rows
        first = torch.empty((n,), dtype=torch.int32, device=self.device)
        last = torch.empty((n,), dtype=torch.int32, device=self.device)
        count, mx = c_int(), c_int()
        self._call(self._lib.pbvi_group_record_blocks(self._h, _ptr(blocks), world, block_rows, words, _ptr(first), _ptr(last), byref(count),
                                                      byref(mx), self._stream))
        return first[:count.value], last[:count.value], mx.value

    def confirm_groups(self, rows: torch.Tensor, first: torch.Tensor, inverse: torch.Tensor) -> bool:
        """True iff every row is bytewise equal to the first row of its group (exactness check of a key-based dedup)."""
        r = _f64(rows, self.device)
        ok = c_int()
        self._call(self._lib.pbvi_confirm_groups(self._h, _ptr(r), r.shape[0], r.shape[1], _ptr(_i32(first, self.device)),
                                                 _ptr(_i32(inverse, self.device)), byref(ok), self._stream))
        return bool(ok.value)

    @staticmethod
    def pack_geometry(row_len: int) -> tuple:
        """(chunks per row, bitmap words per row) of the packed row format."""
        n_c = -(-row_len // 4)
        return n_c, -(-n_c // 32)

    def pack_rows_host(self, rows: torch.Tensor, bitmap: torch.Tensor, row_start: torch.Tensor, packed: torch.Tensor) -> int:
        """Packs host rows [n,L] (float64 CPU tensor) into the given host buffers (pure host code; releases the GIL, so slabs can be
        packed by a thread pool).  Returns the number of 4-double chunks written."""
        n, L = rows.shape
        assert rows.dtype == torch.float64 and rows.is_contiguous() and not rows.is_cuda
        total = c_int64()
        _check(self._lib.pbvi_pack_rows_host(rows.data_ptr(), n, L, bitmap.data_ptr(), row_start.data_ptr(), packed.data_ptr(), byref(total)))
        return int(total.value)

    def unpack_rows(self, bitmap: torch.Tensor, row_start: torch.Tensor, packed: torch.Tensor, out: torch.Tensor,
                    slab_rows: int | None = None, region_chunks: int = 0) -> None:
        """Rebuilds dense rows `out` [n,L] (CUDA float64, contiguous) from device copies of the packed arrays of consecutive slabs
        of `slab_rows` rows (default: one slab), each slab's chunks starting at slab * region_chunks in `packed`."""
        n, L = out.shape
        assert out.is_contiguous() and out.dtype == torch.float64
        self._call(self._lib.pbvi_unpack_rows(self._h, _ptr(bitmap), _ptr(row_start), _ptr(packed), n, L, int(slab_rows or max(n, 1)),
                                              int(region_chunks), _ptr(out), self._stream))

    # ---- packed upload of host-resident rows: persistent staging + packer threads --------------------------------------------
    PACK_SLAB = 64                 # rows packed by one host task (small: the first chunk is ready after a few milliseconds)
    PACK_THREADS = None            # packer threads (None: one per host core but one -- the threads that issue copies and kernels need a core --, at most 32)
    PACK_MAX_DENSITY = 0.6         # above this share of non-zero 4-double chunks the rows are uploaded as they are

    def start_pack(self, host: torch.Tensor):
        """
        Starts packing the pinned host rows [n,L] on the packer threads and returns a job handle (or None when the staging
        buffers are in use by another pending job).  Called when a host-resident BeliefSet is created, so that the host work
        overlaps whatever the caller does before the backup (the upload of the value function, for one);
        `PBVI_Solver._select_streamed` consumes the job: it ships the packed slabs (`_PackJob.shipped`) and unpacks them.
        """
        import os
        import weakref
        from concurrent.futures import ThreadPoolExecutor
        n, L = host.shape
        # Several ranks on one host share its memory bandwidth, and packing adds CPU reads and writes of every byte on top of the
        # DMA traffic: measured at 8 ranks per box it turns a 164 ms end-to-end step into 222 ms, at 2 ranks (11 packer threads each,
        # with the prefetching packer) a 48.8 ms step into 53.8 ms.  One rank per host packs.
        if int(os.environ.get('LOCAL_WORLD_SIZE', '1')) > 1:
            return None
        workers = self.PACK_THREADS or max(1, min(32, (os.cpu_count() or 2) - 1))
        st = self.__dict__.get('_pack')
        if st is not None and st['job'] is not None and st['job']() is not None and not st['job']().consumed:
            return None
        for f in (st or {}).get('futures') or ():  # packers of an abandoned job may still be writing the staging buffers
            f.result()
        if st is not None and st['job'] is not None and st['job']() is None:
            st['stream'].synchronize()             # a job dropped without `close()`: no event marks the end of its copies
        if st is not None and st['copies_done'] is not None:
            st['copies_done'].synchronize()        # the copies of the previous job may still be reading the pinned staging
        if st is None or st['key'] != (n, L) or st['pool']._max_workers != workers:
            n_c, W = self.pack_geometry(L)
            SL = self.PACK_SLAB
            n_slabs = -(-n // SL)
            region = SL * n_c * 4 + 4              # doubles per slab: worst case + the packer's one-chunk slack
            pool = st['pool'] if st is not None and st['pool']._max_workers == workers else ThreadPoolExecutor(max_workers=workers)
            stream = st['stream'] if st is not None else torch.cuda.Stream(device=self.device)
            st = self._pack = {
                'key': (n, L), 'n_c': n_c, 'W': W, 'SL': SL, 'n_slabs': n_slabs, 'region': region, 'pool': pool, 'stream': stream, 'job': None,
                'copies_done': None, 'futures': None, 'alive': None,
                'h_bm': torch.empty((n, W), dtype=torch.int32).pin_memory(),
                'h_rs': torch.empty((n_slabs, SL + 1), dtype=torch.int32).pin_memory(),
                'h_pk': torch.empty((n_slabs * region,), dtype=torch.float64).pin_memory(),
                'd_bm': torch.empty((n, W), dtype=torch.int32, device=self.device),
                'd_rs': torch.empty((n_slabs, SL + 1), dtype=torch.int32, device=self.device),
                'd_pk': torch.empty((n_slabs * region,), dtype=torch.float64, device=self.device)}
        # the unpack kernels of the previous job (the caller's stream waited for each of them) read the device staging the new copies overwrite
        st['stream'].wait_stream(torch.cuda.current_stream(self.device))
        job = _PackJob(self, st, host)
        # the staging dict keeps what the packer threads touch alive for as long as they may run
        st['job'], st['futures'], st['alive'] = weakref.ref(job), job.futures, (job.totals, host)
        return job

    def vi_sweep(self, vopt, gamma: float):
        v = _f64(vopt, self.device)
        assert v.shape == (self.S,)
        alpha = torch.empty((self.A, self.S), dtype=torch.float64, device=self.device)
        vnew = torch.empty((self.S,), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_vi_sweep(self._h, _ptr(v), float(gamma), _ptr(alpha), _ptr(vnew), self._stream))
        return alpha, vnew

    def fib_sweep(self, rows, gamma: float, want_stats: bool = False):
        """One Fast Informed Bound sweep (`pbvi_fib_sweep`): A output rows [A,S] from k input rows [k,S]; with `want_stats` (k == A)
        also the device pair {max(out - rows), max |out - rows|} [2] computed by the same launch."""
        U = self._beliefs(rows)
        out = torch.empty((self.A, self.S), dtype=torch.float64, device=self.device)
        stats = torch.empty((2,), dtype=torch.float64, device=self.device) if want_stats else None
        self._call(self._lib.pbvi_fib_sweep(self._h, _ptr(U), U.shape[0], float(gamma), _ptr(out), _ptr(stats), self._stream))
        return (out, stats) if want_stats else out

    def upper_backup(self, beliefs, fib_rows, gamma: float, corner, idx, val, count, dot, ub_values, n_ub: int, want_action: bool = False):
        """Point-based upper-bound backup of n beliefs (`pbvi_upper_backup`) against the rows `fib_rows` [k,S] and the sawtooth over the
        first n_ub stored beliefs of the support lists: returns (u [n], cur [n]) CUDA float64 tensors (and the maximising action [n] int32
        with `want_action`).  The caller sizes n: the call takes n*A*O*(S + n_ub + 1) doubles of scratch."""
        b, F = self._beliefs(beliefs), self._beliefs(fib_rows)
        n = b.shape[0]
        u = torch.empty((n,), dtype=torch.float64, device=self.device)
        cur = torch.empty((n,), dtype=torch.float64, device=self.device)
        act = torch.empty((n,), dtype=torch.int32, device=self.device) if want_action else None
        on = n_ub > 0
        self._call(self._lib.pbvi_upper_backup(self._h, _ptr(b), n, _ptr(F), F.shape[0], float(gamma), _ptr(corner), _ptr(idx) if on else None,
                                               _ptr(val) if on else None, _ptr(count) if on else None, _ptr(dot) if on else None,
                                               _ptr(ub_values) if on else None, int(n_ub), _ptr(u), _ptr(cur), _ptr(act), self._stream))
        return (u, cur, act) if want_action else (u, cur)

    def prune_dominated(self, alphas) -> torch.Tensor:
        al = self._beliefs(alphas)
        keep = torch.empty((al.shape[0],), dtype=torch.int32, device=self.device)
        self._call(self._lib.pbvi_prune_dominated(self._h, _ptr(al), al.shape[0], _ptr(keep), self._stream))
        return keep

    def prune_lp(self, alphas):
        """LP-domination prune of pairwise distinct rows (see `pbvi_prune_lp`): returns (keep [n] int32 CUDA tensor, bound [n] float64
        CUDA tensor, counts int64 [4] = {kept at a corner, kept by an LP witness, pruned, kept undecided}).  Synchronises."""
        al = self._beliefs(alphas)
        n = al.shape[0]
        keep = torch.empty((n,), dtype=torch.int32, device=self.device)
        bound = torch.empty((n,), dtype=torch.float64, device=self.device)
        counts = np.zeros(4, dtype=np.int32)
        self._call(self._lib.pbvi_prune_lp(self._h, _ptr(al), n, _ptr(keep), _ptr(bound), counts.ctypes.data, self._stream))
        return keep, bound, counts.astype(np.int64)

    def prune_lp_certificates(self, alphas):
        """`prune_lp` that also returns the certificate of every pruned row (`pbvi_prune_lp_certificates`): (keep, bound, counts, idx
        [n, 64] int32, weights [n, 64] float64), idx / weights the competitor set J (-1 padded) and the lambda of the verified bound u
        (0 padded); -1 / 0 throughout for a kept row.  Synchronises."""
        al = self._beliefs(alphas)
        n = al.shape[0]
        keep = torch.empty((n,), dtype=torch.int32, device=self.device)
        bound = torch.empty((n,), dtype=torch.float64, device=self.device)
        idx = torch.empty((n, 64), dtype=torch.int32, device=self.device)
        w = torch.empty((n, 64), dtype=torch.float64, device=self.device)
        counts = np.zeros(4, dtype=np.int32)
        self._call(self._lib.pbvi_prune_lp_certificates(self._h, _ptr(al), n, _ptr(keep), _ptr(bound), counts.ctypes.data, _ptr(idx), _ptr(w),
                                                        self._stream))
        return keep, bound, counts.astype(np.int64), idx, w

    def prune_lp_stats(self) -> dict:
        """Work of the last `prune_lp` call: largest competitor set, restricted LPs, simplex pivots, rows that reached the LP stage."""
        out = np.zeros(4, dtype=np.int64)
        _check(self._lib.pbvi_prune_lp_stats(self._h, out.ctypes.data))
        return dict(max_competitors=int(out[0]), lps=int(out[1]), pivots=int(out[2]), lp_rows=int(out[3]))

    def bpi_lp(self, pool, n: int, tau: float, corner, price, cols, ncols, bstar, delta, u, lam, mstar, status) -> dict:
        """One round of the restricted master LPs of bounded policy iteration (`pbvi_bpi_lp`) on n entries, updating the state tensors in
        place: pool [P, S] float64 (rows 0..n-1 the node rows, rows n..2n-1 their own one-sweep rows, then priced columns), corner / price /
        ncols / status int32 [n], cols int32 [n, 64], bstar float64 [n, S], delta / u / mstar float64 [n], lam float64 [n, 64], all CUDA and
        contiguous.  Returns {max_columns, lps, pivots, entries}.  Synchronises."""
        S = self.S
        for t, shape, dt in ((pool, (pool.shape[0], S), torch.float64), (corner, (n,), torch.int32), (price, (n,), torch.int32),
                             (cols, (n, 64), torch.int32), (ncols, (n,), torch.int32), (bstar, (n, S), torch.float64),
                             (delta, (n,), torch.float64), (u, (n,), torch.float64), (lam, (n, 64), torch.float64),
                             (mstar, (n,), torch.float64), (status, (n,), torch.int32)):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dt and tuple(t.shape) == shape and t.is_contiguous()):
                raise ValueError(f'bpi_lp: expected a contiguous CUDA {dt} tensor of shape {shape}')
        act = status == -1
        if bool(act.any()):
            k = ncols[act]
            listed = torch.arange(64, device=self.device)[None, :] < ncols[act][:, None].long()
            c, p, s0 = cols[act][listed], price[act], corner[act]
            if (int(k.min()) < 1 or int(k.max()) > 64 or int(c.min()) < 0 or int(c.max()) >= pool.shape[0] or int(p.max()) >= pool.shape[0]
                    or int(s0.min()) < 0 or int(s0.max()) >= S):
                raise ValueError('bpi_lp: active entries need 1..64 columns, column and price rows below the pool size and corners in [0, S)')
        out = np.zeros(4, dtype=np.int64)
        self._call(self._lib.pbvi_bpi_lp(self._h, _ptr(pool), pool.shape[0], int(n), float(tau), _ptr(corner), _ptr(price), _ptr(cols),
                                         _ptr(ncols), _ptr(bstar), _ptr(delta), _ptr(u), _ptr(lam), _ptr(mstar), _ptr(status),
                                         out.ctypes.data, self._stream))
        return dict(max_columns=int(out[0]), lps=int(out[1]), pivots=int(out[2]), entries=int(out[3]))

    def _finite_rows(self, rows, what: str) -> torch.Tensor:
        X = self._beliefs(rows)
        if X.shape[0] and not bool(torch.isfinite(X).all()):
            raise ValueError(f'{what}: rows must be finite')
        return X

    def ip_project(self, alphas, gamma: float, action: int) -> torch.Tensor:
        """The projections of incremental pruning (`pbvi_ip_project`): G [O, nV, S] CUDA float64, G[o, v] = gamma * sum_r RTO[:, a, o, r] *
        alpha_v[reach[:, a, r]], bitwise the term `backup_assemble` forms for observation o.  The rows must be finite."""
        al = self._finite_rows(alphas, 'ip_project')
        if not 0 <= int(action) < self.A:
            raise ValueError(f'ip_project: action must lie in [0, {self.A})')
        out = torch.empty((self.O, al.shape[0], self.S), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_ip_project(self._h, _ptr(al), al.shape[0], float(gamma), int(action), _ptr(out), self._stream))
        return out

    def ip_cross_sum(self, x, g, action: int = -1) -> torch.Tensor:
        """The cross sum of incremental pruning (`pbvi_ip_cross_sum`): rows x_i + g_j [nx * ng, S] (i-major), with action >= 0 Rbar[:, a] +
        (x_i + g_j); x = None gives g_j (or Rbar[:, a] + g_j)."""
        G = self._beliefs(g)
        X = None if x is None else self._beliefs(x)
        if not -1 <= int(action) < self.A:
            raise ValueError(f'ip_cross_sum: action must lie in [-1, {self.A})')
        nx = 1 if X is None else X.shape[0]
        out = torch.empty((nx * G.shape[0], self.S), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_ip_cross_sum(self._h, _ptr(X), 0 if X is None else X.shape[0], _ptr(G), G.shape[0], int(action), _ptr(out),
                                               self._stream))
        return out

    def ip_residual_lp(self, new_rows, old_rows, tau: float) -> dict:
        """How far each row y_i of `new_rows` rises above the rows of `old_rows` (`pbvi_ip_residual_lp`), delta_i = max_b min_j b . (y_i - x_j):
        {u [ny] (verified upper bound), mstar [ny] (lower bound), bstar [ny, S], cert_idx [ny, 64] int32, cert_w [ny, 64], stats} as CUDA
        tensors, stats = {max_competitors, lps, pivots, budget_rows}.  Rows must be finite and old_rows non-empty.  Synchronises."""
        Y, X = self._finite_rows(new_rows, 'ip_residual_lp'), self._finite_rows(old_rows, 'ip_residual_lp')
        if X.shape[0] < 1:
            raise ValueError('ip_residual_lp: need at least one old row')
        if not (tau >= 0.0 and np.isfinite(tau)):
            raise ValueError('ip_residual_lp: tau must be finite and >= 0')
        ny = Y.shape[0]
        u, mstar = (torch.empty((ny,), dtype=torch.float64, device=self.device) for _ in range(2))
        bstar = torch.empty((ny, self.S), dtype=torch.float64, device=self.device)
        idx = torch.empty((ny, 64), dtype=torch.int32, device=self.device)
        w = torch.empty((ny, 64), dtype=torch.float64, device=self.device)
        st = np.zeros(4, dtype=np.int64)
        self._call(self._lib.pbvi_ip_residual_lp(self._h, _ptr(Y), ny, _ptr(X), X.shape[0], float(tau), _ptr(u), _ptr(mstar), _ptr(bstar),
                                                 _ptr(idx), _ptr(w), st.ctypes.data, self._stream))
        return dict(u=u, mstar=mstar, bstar=bstar, cert_idx=idx, cert_w=w,
                    stats=dict(max_competitors=int(st[0]), lps=int(st[1]), pivots=int(st[2]), budget_rows=int(st[3])))

    def sawtooth(self, corner, ub_beliefs, ub_values, queries) -> torch.Tensor:
        c, q = _f64(corner, self.device), self._beliefs(queries)
        ubb = _f64(ub_beliefs, self.device).reshape(-1, self.S)
        ubv = _f64(ub_values, self.device).reshape(-1)
        out = torch.empty((q.shape[0],), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_sawtooth(self._h, _ptr(c), _ptr(ubb) if ubb.shape[0] else None, _ptr(ubv) if ubb.shape[0] else None,
                                       ubb.shape[0], _ptr(q), q.shape[0], _ptr(out), self._stream))
        return out

    def support_lists(self, rows: torch.Tensor, corner: torch.Tensor, idx: torch.Tensor, val: torch.Tensor, count: torch.Tensor,
                      dot: torch.Tensor) -> None:
        """Support lists (states / values of the positive entries, ELL layout with row pitch S) and row . corner of `rows` [n,S], written
        into the given slices (idx int32 [n,S], val f64 [n,S], count int32 [n], dot f64 [n])."""
        n = rows.shape[0]
        assert rows.is_contiguous() and idx.is_contiguous() and val.is_contiguous() and idx.shape == (n, self.S) and val.shape == (n, self.S)
        self._call(self._lib.pbvi_support_lists(self._h, _ptr(rows), n, _ptr(corner), _ptr(idx), _ptr(val), _ptr(count), _ptr(dot), self._stream))

    def sawtooth_lists(self, corner, idx, val, count, dot, ub_values, n_ub: int, queries) -> torch.Tensor:
        q = self._beliefs(queries)
        out = torch.empty((q.shape[0],), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_sawtooth_lists(self._h, _ptr(corner), _ptr(idx), _ptr(val), _ptr(count), _ptr(dot), _ptr(ub_values), int(n_ub),
                                                 _ptr(q), q.shape[0], _ptr(out), self._stream))
        return out

    def sawtooth_witness(self, corner, idx, val, count, dot, ub_values, n_ub: int) -> tuple:
        """Sawtooth dominance among the n_ub stored pairs of the support lists (`pbvi_sawtooth_witness`): returns (min [n_ub] f64 =
        min_{j != i} s_j(b_i), arg [n_ub] int32 = its first j or -1 when no term lies below v0(b_i), self [n_ub] f64 = s_i(b_i))."""
        n_ub = int(n_ub)
        mn = torch.empty((n_ub,), dtype=torch.float64, device=self.device)
        arg = torch.empty((n_ub,), dtype=torch.int32, device=self.device)
        own = torch.empty((n_ub,), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_sawtooth_witness(self._h, _ptr(corner), _ptr(idx), _ptr(val), _ptr(count), _ptr(dot), _ptr(ub_values), n_ub,
                                                   _ptr(mn), _ptr(arg), _ptr(own), self._stream))
        return mn, arg, own

    def hsvi_level(self, b: torch.Tensor, alphas: torch.Tensor, gamma: float, corner, idx, val, count, dot, ub_values, n_ub: int,
                   stored_keys, stored_vals, n_stored: int, conv_term: float, may_continue: bool, next_out: torch.Tensor | None = None,
                   want_successors: bool = True):
        """One level of HSVI's exploration (`pbvi_hsvi_level`): returns (successors [A,O,S] | None, masses [A,O] | None,
        (best_a, best_o, Q, upper - lower), (added, key0, key1, n_possible)); the chosen successor is written into `next_out` [S]."""
        al = alphas if (isinstance(alphas, torch.Tensor) and alphas.is_cuda and alphas.is_contiguous() and alphas.dtype == torch.float64) else self._beliefs(alphas)
        succ = mass = None
        if want_successors:
            succ = torch.empty((self.A, self.O, self.S), dtype=torch.float64, device=self.device)
            mass = torch.empty((self.A, self.O), dtype=torch.float64, device=self.device)
        out = np.empty(8, dtype=np.float64)
        cap = 0 if stored_keys is None else stored_keys.shape[0]
        self._call(self._lib.pbvi_hsvi_level(self._h, _ptr(b), _ptr(al), al.shape[0], float(gamma), _ptr(corner), _ptr(idx), _ptr(val), _ptr(count),
                                             _ptr(dot), _ptr(ub_values), int(n_ub), _ptr(stored_keys), _ptr(stored_vals), int(n_stored), int(cap),
                                             float(conv_term), int(bool(may_continue)), _ptr(next_out), _ptr(succ), _ptr(mass), out.ctypes.data,
                                             self._stream))
        return succ, mass, out[:4], out[4:].view(np.int64)

    def gap_trial_step(self, beliefs, lower_rows, fib_rows, gamma: float, corner, idx, val, count, dot, ub_values, n_ub: int, theta: float,
                       uniforms=None, want_bounds: bool = False):
        """One level of K gap-driven trials (`pbvi_gap_trial_step`): returns (out [K,4] CUDA float64 = {a*, o*, Q*, e_{o*}} per trial, next
        beliefs [K,S]), and with `want_bounds` also (U [K,O], L [K,O]).  `uniforms` [K] (None: the argmax rule everywhere; a negative
        entry: the argmax rule for that trial).  The caller sizes K: the call takes K*A*O*(S + n_ub + 1) doubles of scratch."""
        b, X, F = self._beliefs(beliefs), self._beliefs(lower_rows), self._beliefs(fib_rows)
        K = b.shape[0]
        u = None if uniforms is None else _f64(uniforms, self.device).reshape(-1)
        assert u is None or u.shape == (K,)
        out = torch.empty((K, 4), dtype=torch.float64, device=self.device)
        nxt = torch.empty((K, self.S), dtype=torch.float64, device=self.device)
        U = torch.empty((K, self.O), dtype=torch.float64, device=self.device) if want_bounds else None
        L = torch.empty((K, self.O), dtype=torch.float64, device=self.device) if want_bounds else None
        on = n_ub > 0
        self._call(self._lib.pbvi_gap_trial_step(self._h, _ptr(b), K, _ptr(X), X.shape[0], _ptr(F), F.shape[0], float(gamma), _ptr(corner),
                                                 _ptr(idx) if on else None, _ptr(val) if on else None, _ptr(count) if on else None,
                                                 _ptr(dot) if on else None, _ptr(ub_values) if on else None, int(n_ub), float(theta), _ptr(u),
                                                 _ptr(out), _ptr(nxt), _ptr(U), _ptr(L), self._stream))
        return (out, nxt, U, L) if want_bounds else (out, nxt)

    def min_l2_distance(self, beliefs, candidates) -> torch.Tensor:
        b, c = self._beliefs(beliefs), self._beliefs(candidates)
        out = torch.empty((c.shape[0],), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_min_l2_distance(self._h, _ptr(b), b.shape[0], _ptr(c), c.shape[0], _ptr(out), self._stream))
        return out

    def ger_scores(self, beliefs, alpha_b, successors, r_min: float, r_max: float) -> torch.Tensor:
        """GER error terms eps[n,A,O] (reference src/pomdp.py:1738-1748)."""
        b, al = self._beliefs(beliefs), self._beliefs(alpha_b)
        sc = _f64(successors, self.device)
        n = b.shape[0]
        assert al.shape == b.shape and sc.shape == (n, self.A, self.O, self.S)
        eps = torch.empty((n, self.A, self.O), dtype=torch.float64, device=self.device)
        self._call(self._lib.pbvi_ger_scores(self._h, _ptr(b), _ptr(al), _ptr(sc), n, float(r_min), float(r_max), _ptr(eps), self._stream))
        return eps

    def _staging_buffer(self, n: int) -> torch.Tensor:
        """Grow-only pinned staging of the read-backs; every new use invalidates the views handed out before (`_staging_token`)."""
        stream = getattr(self, '_readback_stream', None)
        if stream is not None:
            stream.synchronize()                    # an abandoned mirror may still be writing the staging
        buf = getattr(self, '_staging', None)
        want = max(n, getattr(self, '_staging_want', 0), 1 << 20)
        if buf is None or buf.numel() < n:
            buf = self._staging = torch.empty((want,), dtype=torch.float64).pin_memory()
        self._staging_token = getattr(self, '_staging_token', 0) + 1
        return buf

    def to_host_staged(self, t: torch.Tensor) -> np.ndarray:
        """Device -> host through a grow-only pinned staging buffer; returns a NumPy view valid until the next call."""
        n = t.numel()
        view = self._staging_buffer(n)[:n].view(t.shape)
        view.copy_(t)
        return view.numpy()

    def mirror_begin(self, rows: torch.Tensor) -> dict:
        """
        Starts reading `rows` [n,L] (complete on the current stream) back into the pinned staging on the read-back stream and returns
        a handle for `mirror_finish`.  The streamed backup uses it for the alpha rows it can assemble before its last chunk of beliefs
        is selected: their device->host copy then runs beside the score kernel instead of after it (the link is full duplex).
        """
        n = rows.numel()
        buf = self._staging_buffer(max(2 * n, n + 512 * rows.shape[1]))     # room for the rows the last chunk may add
        stream = getattr(self, '_readback_stream', None)
        if stream is None:
            stream = self._readback_stream = torch.cuda.Stream(device=self.device)
        stream.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(stream):
            buf[:n].view(rows.shape).copy_(rows, non_blocking=True)
        return {'buf': buf, 'token': self._staging_token, 'rows': rows.shape[0], 'L': rows.shape[1], 'stream': stream, 'keep': rows}

    def mirror_finish(self, mirror: dict, tail: torch.Tensor | None):
        """
        Appends `tail` [m,L] (complete on the current stream; None: nothing to add) to the read-back started by `mirror_begin`.
        Returns (NumPy view of all rows, CUDA event behind the copies, staging token), or None when the staging was re-used in
        between or is too small (the next one is allocated larger; the caller reads the rows back the plain way).
        """
        n0, L = mirror['rows'], mirror['L']
        m = 0 if tail is None else tail.shape[0]
        buf, stream = mirror['buf'], mirror['stream']
        if mirror['token'] != getattr(self, '_staging_token', 0):
            return None
        if (n0 + m) * L > buf.numel():
            self._staging_want = 2 * (n0 + m) * L
            return None
        if m:
            stream.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(stream):
                buf[n0 * L:(n0 + m) * L].view(m, L).copy_(tail, non_blocking=True)
        done = torch.cuda.Event()
        done.record(stream)
        return buf[:(n0 + m) * L].view(n0 + m, L).numpy(), done, mirror['token']

    def set_option(self, name: str, value: int) -> None:
        _check(self._lib.pbvi_set_option(self._h, name.encode(), int(value)))

    def set_profiling(self, enable: bool) -> None:
        _check(self._lib.pbvi_set_profiling(self._h, int(enable)))

    def last_score_ms(self) -> float:
        ms = ctypes.c_float()
        _check(self._lib.pbvi_last_score_ms(self._h, byref(ms)))
        return float(ms.value)

    def last_stats(self) -> dict:
        e, d, n = c_double(), c_double(), c_int()
        _check(self._lib.pbvi_last_stats(self._h, byref(e), byref(d), byref(n)))
        return dict(executed_flops=e.value, dense_flops=d.value, launches=n.value)


class _PackJob:
    """
    Packed upload of host rows in flight.  The packer threads each make ONE library call (slabs t, t + T, t + 2T, ... in a C loop, GIL
    released throughout) and publish a slab's chunk count as their last store; `result(i)` = number of chunks of slab i (waits until it
    is packed).  `shipped(rows)` follows the packers slab by slab, enqueues the copies [chunks of every slab | bitmaps | row offsets]
    of the ship units up to `rows` on the upload stream and returns the CUDA event behind them; the consumer makes its stream wait on
    it and unpacks.  A ship unit is one round of the packer threads (T slabs, at most SHIP_SLABS), so the first one is complete after
    ONE slab time.  (A feeder thread that ships while the caller is still busy elsewhere was measured: no gain, the link is taken by
    the value function's upload until the caller is back; tools/e2e_timeline.py.)
    """
    SHIP_SLABS = 16

    def __init__(self, dev: 'DeviceModel', st: dict, host: torch.Tensor):
        self.st, self.host, self.consumed = st, host, False
        n, L = host.shape
        self.n = n
        self.totals = np.full((st['n_slabs'],), -1, dtype=np.int64)
        lib, pool = dev._lib, st['pool']
        T = max(1, min(pool._max_workers, st['n_slabs']))
        self.ship_rows = st['SL'] * min(T, self.SHIP_SLABS)
        args = (host.data_ptr(), n, L, st['SL'])
        tail = (st['h_bm'].data_ptr(), st['h_rs'].data_ptr(), st['h_pk'].data_ptr(), st['region'], self.totals.ctypes.data)
        self.futures = [pool.submit(lib.pbvi_pack_slabs_host, *args, t, T, *tail) for t in range(T)]
        self.max_density = dev.PACK_MAX_DENSITY
        self.events = [None] * (-(-n // self.ship_rows))     # CUDA event behind the copies of ship unit u
        self.units_shipped = 0
        self.h2d_bytes = 0

    def result(self, i: int) -> int:
        import time
        while True:
            v = int(self.totals[i])
            if v >= 0:
                return v
            if v == -2 or all(f.done() for f in self.futures) and int(self.totals[i]) < 0:
                raise PBVIError('packing the host rows failed')
            time.sleep(2e-5)

    def is_packed(self) -> bool:
        """Sparse enough to travel packed (decided on the first slab)?  False: nothing is shipped, the caller copies the rows."""
        st = self.st
        return self.result(0) <= self.max_density * min(st['SL'], self.n) * st['n_c']

    def shipped(self, rows: int):
        """CUDA event behind the copies of the first `rows` rows (ships every unit up to there that is not on its way yet)."""
        st, n = self.st, self.n
        SL, region, W, stream = st['SL'], st['region'], st['W'], st['stream']
        units = -(-rows // self.ship_rows)
        with torch.cuda.stream(stream):
            while self.units_shipped < units:
                u = self.units_shipped
                lo, hi = u * self.ship_rows, min(n, (u + 1) * self.ship_rows)
                s0, s1 = lo // SL, -(-hi // SL)
                for i in range(s0, s1):
                    total = self.result(i)                               # the packers run ahead of the copies
                    st['d_pk'][i * region:i * region + total * 4].copy_(st['h_pk'][i * region:i * region + total * 4], non_blocking=True)
                    self.h2d_bytes += total * 32
                st['d_bm'][lo:hi].copy_(st['h_bm'][lo:hi], non_blocking=True)
                st['d_rs'][s0:s1].copy_(st['h_rs'][s0:s1], non_blocking=True)
                self.h2d_bytes += (hi - lo) * W * 4 + (s1 - s0) * (SL + 1) * 4
                self.events[u] = torch.cuda.Event(enable_timing=True)
                self.events[u].record(stream)
                self.units_shipped = u + 1
        return self.events[units - 1]

    def close(self) -> None:
        """The consumer is done with the job (or never used it): the staging buffers become free once the enqueued copies have run."""
        if not self.consumed:
            self.consumed = True
            done = torch.cuda.Event()
            done.record(self.st['stream'])
            self.st['copies_done'] = done
