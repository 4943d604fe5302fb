"""
AlphaVector / ValueFunction with the reference's interface (src/mdp.py:593-1278) on device-resident storage.

`alpha_vector_array` is a CUDA float64 torch tensor [N,S] (the reference's GPU path holds a CuPy array there),
`actions` a host int64 array.  Construction de-duplicates on the raw bytes of the rows exactly like the reference's
`{values.tobytes(): alpha_vector}` dict -- position of the first occurrence, action of the last -- and `extend` is the
same dict `update` (new rows first, the other side's action wins on a collision); both run through `sets.dedup_rows`.
"""
from __future__ import annotations

import os
import itertools
from datetime import datetime
from typing import Union

import numpy as np
import torch

from .model import Model, log
from .sets import dedup_rows


_UID = itertools.count(1)


class AlphaVector:
    """A vector over states with the action it belongs to (reference src/mdp.py:593-610)."""

    def __init__(self, values, action: int) -> None:
        self.values = values
        self.action = int(action)


def _rows_to_device(model: Model, rows) -> torch.Tensor:
    dev = model.device.device
    if isinstance(rows, torch.Tensor):
        return rows.to(device=dev, dtype=torch.float64).contiguous()
    return torch.as_tensor(np.ascontiguousarray(rows, dtype=np.float64)).to(dev)


class ValueFunction:
    """
    Set of alpha vectors approximating the value function (reference src/mdp.py:612-1278).

    Parameters
    ----------
    model : Model
    alpha_vectors : list[AlphaVector] | np.ndarray | torch.Tensor, optional
    action_list : list[int] | np.ndarray, optional
        Actions of the rows when `alpha_vectors` is an array.
    """

    def __init__(self, model: Model, alpha_vectors: Union[list, np.ndarray, torch.Tensor] = [], action_list=[], *,
                 _trusted: bool = False, _hashes: np.ndarray | None = None):
        self.model = model
        self.is_on_gpu = True
        self._pruning_level = 1
        self.uid = next(_UID)               # identity of this row set for per-belief result caches (solver.compute_change)
        self.parent_uid = None              # set by PBVI_Solver.backup(append=True): rows == first `n_new` rows + every parent row
        self.n_new = 0
        S = model.state_count
        if isinstance(alpha_vectors, list):
            assert all(v.values.shape[0] == S for v in alpha_vectors), \
                f"Some or all alpha vectors in the list provided dont have the right size, they should be of shape: {S}"
            actions = np.array([v.action for v in alpha_vectors], dtype=np.int64)
            if len(alpha_vectors):
                rows = torch.stack([_rows_to_device(model, v.values) for v in alpha_vectors])
            else:
                rows = torch.empty((0, S), dtype=torch.float64, device=model.device.device)
        else:
            actions = np.asarray(action_list.cpu() if isinstance(action_list, torch.Tensor) else action_list).astype(np.int64).reshape(-1)
            av_shape, exp_shape = tuple(alpha_vectors.shape), (len(actions), S)
            assert av_shape == exp_shape, f"Alpha vector array does not have the right shape (received: {av_shape}; expected: {exp_shape})"
            rows = _rows_to_device(model, alpha_vectors)
        if _trusted:
            self._array, self._actions, self._hashes = rows, actions, _hashes
        else:
            first, last, hashes, _ = dedup_rows(model.device, rows)
            if first.shape[0] == rows.shape[0]:
                self._array, self._actions, self._hashes = rows, actions, hashes
            else:
                self._array = rows[torch.as_tensor(first, device=rows.device)]
                self._actions, self._hashes = actions[last], hashes[first]
        self._vector_list = None

    # ---- reference attributes ------------------------------------------------------------------
    @property
    def alpha_vector_array(self) -> torch.Tensor:
        """[N,S] CUDA float64 tensor."""
        return self._array

    @property
    def actions(self) -> np.ndarray:
        return self._actions

    @property
    def alpha_vector_list(self) -> list:
        if self._vector_list is None:
            self._vector_list = [AlphaVector(row, a) for row, a in zip(self._array, self._actions)]
        return self._vector_list

    @property
    def row_hashes(self) -> np.ndarray:
        if self._hashes is None:
            self._hashes = self.model.device.row_hash(self._array).cpu().numpy() if len(self) else np.zeros((0, 2), dtype=np.int64)
        elif isinstance(self._hashes, torch.Tensor):              # keys left on the device by the backup: fetched on first use
            self._hashes = self._hashes.cpu().numpy()
        return self._hashes

    def __len__(self) -> int:
        return int(self._array.shape[0])

    def numpy(self, staged: bool = False):
        """
        (alpha_vector_array, actions) as host NumPy arrays.  `staged=True` reads the rows back through the model's
        reusable pinned staging buffer and returns a VIEW of it (valid until the next staged read): a device->host copy at
        PCIe speed without a fresh pageable allocation per call.
        """
        if staged:
            mirror = self.__dict__.get('_mirror')       # the streamed backup read the rows back while it was still computing
            if mirror is not None and mirror[0].shape[0] == len(self) and mirror[2] == getattr(self.model.device, '_staging_token', 0):
                mirror[1].synchronize()
                return mirror[0], self._actions.copy()
            return self.model.device.to_host_staged(self._array), self._actions.copy()
        return self._array.cpu().numpy(), self._actions.copy()

    # ---- set operations --------------------------------------------------------------------------
    def _union(self, other: 'ValueFunction') -> tuple:
        fast = self._union_prepend(other)
        if fast is not None:
            return fast
        rows = torch.cat([self._array, other._array], dim=0)
        actions = np.concatenate([self._actions, other._actions])
        hashes = np.concatenate([self.row_hashes, other.row_hashes], axis=0)
        first, last, _, _ = dedup_rows(self.model.device, rows, hashes)
        if first.shape[0] != rows.shape[0]:
            rows = rows[torch.as_tensor(first, device=rows.device)]
        return rows, actions[last], hashes[first], None

    def _union_prepend(self, other: 'ValueFunction'):
        """
        The solve loop's case -- a few new rows in front of a large, disjoint old set -- without copying the old rows: they
        live at the END of a front-growing buffer and the new rows are written just before them, so the union is the view
        [new rows | old rows] and the old value function keeps viewing its own suffix (rows are never mutated).
        Returns None (general path) when any key occurs twice or the buffer is shared with another descendant.
        """
        n_self, n_other = len(self), len(other)
        if n_self == 0 or n_other == 0:
            return None
        hashes = np.concatenate([self.row_hashes, other.row_hashes], axis=0)
        # all keys distinct?  Checked on a 64-bit mix of the two halves with one SIMD sort (0.1 ms at 9000 rows; a set of Python
        # tuples costs 5 ms there, every backup of a long solve): distinct mixes imply distinct keys, and a repeated mix -- a real
        # duplicate or a 2^-64 accident -- just takes the general path below.
        with np.errstate(over='ignore'):
            mix = np.sort(hashes[:, 0] ^ (hashes[:, 1] * np.int64(-7046029254386353131)))
        if np.any(mix[1:] == mix[:-1]):
            return None
        S = self.model.state_count
        buf, start = other.__dict__.get('_buf'), other.__dict__.get('_buf_start')
        shared = other.__dict__.get('_buf_front')          # [smallest start handed out so far] shared by every view of the buffer
        if buf is None or shared[0] != start or start < n_self:
            cap = 2 * (n_self + n_other) + 64
            buf = torch.empty((cap, S), dtype=torch.float64, device=self._array.device)
            start = cap - n_other
            buf[start:] = other._array
            shared = [start]
        buf[start - n_self:start] = self._array
        shared[0] = start - n_self
        rows = buf[start - n_self:start + n_other]
        return rows, np.concatenate([self._actions, other._actions]), hashes, (buf, start - n_self, shared)

    def __add__(self, other: 'ValueFunction') -> 'ValueFunction':
        rows, actions, hashes, buf = self._union(other)
        out = ValueFunction(self.model, rows, actions, _trusted=True, _hashes=hashes)
        if buf is not None:
            out._buf, out._buf_start, out._buf_front = buf
        return out

    def extend(self, other: 'ValueFunction') -> None:
        """In-place union (reference src/mdp.py:763-779): own rows first, then the unseen rows of `other`; on a byte
        collision the other side's action replaces ours."""
        self._array, self._actions, self._hashes, buf = self._union(other)
        self._buf, self._buf_start, self._buf_front = buf if buf is not None else (None, None, None)
        self._vector_list = None
        self._pruning_level = 1
        self._mirror = None
        self.uid, self.parent_uid, self.n_new = next(_UID), None, 0

    def append(self, alpha_vector: AlphaVector) -> None:
        """Adds one alpha vector without de-duplication (reference src/mdp.py:739-760)."""
        assert alpha_vector.values.shape[0] == self.model.state_count, \
            f"Vector to add to value function doesn't have the right size (received: {alpha_vector.values.shape[0]}, expected: {self.model.state_count})"
        row = _rows_to_device(self.model, alpha_vector.values)[None, :]
        self._array = torch.cat([self._array, row], dim=0)
        self._actions = np.append(self._actions, alpha_vector.action)
        self._hashes = None
        self._vector_list = None
        self._mirror = None
        self.uid, self.parent_uid, self.n_new = next(_UID), None, 0
        self._buf = None

    def to_gpu(self) -> 'ValueFunction':
        return self

    def to_cpu(self) -> 'ValueFunction':
        """Kept for interface compatibility: storage is always device-resident; use `.numpy()` for host arrays."""
        return self

    # ---- pruning -------------------------------------------------------------------------------
    def prune(self, level: int = 1) -> None:
        """
        Level 1 is a no-op (duplicates never enter).  Level 2 removes pointwise-dominated vectors (reference src/mdp.py:857-866).

        Level 3 first runs level 2, then removes the vectors that a convex combination of the others beats everywhere -- the LP
        domination the reference intended (src/mdp.py:834-906; its branch fails on the undefined `pruned_alpha_set` at :872).  With
        tau = 1e-9 * max(1, max |alpha|), alpha_i is removed only with a certificate: weights lambda >= 0 summing to 1 over the other
        rows with sum_j lambda_j alpha_j[s] > alpha_i[s] + tau at every state, re-checked in FP64 from the rows.  Every other row
        stays: rows with a witness belief (alpha_i . b - max_{j != i} alpha_j . b > -tau), near-ties, rows whose search ran out of
        budget, and rows with a non-finite entry.  A removed row lies more than tau below another row at every belief, and following
        the rows that beat it ends at a kept row, so max_v alpha_v . b over the kept rows equals the max over all rows at every
        belief.  Kept rows keep their order, actions and row hashes; pruning the result again removes nothing.
        """
        if level < self._pruning_level or level > 3:
            log('Attempting to prune a value function to a level already reached. Returning \'self\'')
            return
        if level >= 2 and self._pruning_level < 2 and len(self) > 0:
            self._select_rows(self.model.device.prune_dominated(self._array))
        if level >= 3 and self._pruning_level < 3 and len(self) > 0:
            self._select_rows(self.model.device.prune_lp(self._array)[0])
        self._pruning_level = level

    def _select_rows(self, keep: torch.Tensor) -> None:
        """Keeps the rows flagged in `keep` (device int32 [n]) in their order, with their actions and hashes."""
        idx = np.flatnonzero(keep.cpu().numpy())
        self._array = self._array[torch.as_tensor(idx, device=self._array.device)]
        self._actions = self._actions[idx]
        self._hashes = None if self._hashes is None else self.row_hashes[idx]
        self._vector_list = None
        self._mirror = None
        self.uid, self.parent_uid, self.n_new = next(_UID), None, 0
        self._buf = None

    # ---- persistence (reference src/mdp.py:909-1036): column 0 `action`, then one column per state label ----------
    def _frame(self, path):
        import pandas as pd
        if not os.path.exists(path):
            print('Folder does not exist yet, creating it...')
            os.makedirs(path)
        rows, actions = self.numpy()
        data = np.concatenate((actions[:, None], rows), axis=1)
        return pd.DataFrame(data, columns=['action', *self.model.state_labels])

    def save(self, path: str = './ValueFunctions', file_name: Union[str, None] = None, compress: bool = False) -> None:
        df = self._frame(path)
        if file_name is None:
            file_name = datetime.now().strftime('%Y%m%d_%H%M%S') + '_value_function.csv'
        if '.csv' not in file_name:
            file_name += '.csv'
        compression_type = None
        if compress:
            file_name += '.gzip'
            compression_type = 'gzip'
        df.to_csv(path + '/' + file_name, index=False, compression=compression_type)

    def save_parquet(self, path: str = './ValueFunctions', file_name: Union[str, None] = None) -> None:
        df = self._frame(path)
        if file_name is None:
            file_name = datetime.now().strftime('%Y%m%d_%H%M%S') + '_value_function.parquet'
        if '.parquet' not in file_name:
            file_name += '.parquet'
        df.to_parquet(path + '/' + file_name, index=False)

    @classmethod
    def load_from_file(cls, file: str, model: Model) -> 'ValueFunction':
        import pandas as pd
        compression_type = 'gzip' if '.gzip' in file else None
        data = pd.read_csv(file, header=0, index_col=False, compression=compression_type).to_numpy()
        return ValueFunction(model, alpha_vectors=data[:, 1:], action_list=data[:, 0].astype(int))

    @classmethod
    def load_from_parquet(cls, file: str, model: Model) -> 'ValueFunction':
        import pandas as pd
        data = pd.read_parquet(file).to_numpy()
        return ValueFunction(model, alpha_vectors=data[:, 1:], action_list=data[:, 0].astype(int))
