"""
B200-native PBVI backup engine: a drop-in for the solver of PimLb/POMDP_PBVI_Exploration (`src/pomdp.py`).

Same names as the reference -- `Model`, `Belief`, `BeliefSet`, `AlphaVector`, `ValueFunction`, `PBVI_Solver`,
`HSVI_Solver`, `FSVI_Solver`, `FSVI_EG_Solver`, `VI_Solver`, `BeliefValueMapping`, `SolverHistory`, `Agent`, `Simulation`,
`SimulationSet` -- plus certified upper bounds on V* (`FIB_Solver`, `UpperBound`) and finite-state controllers evaluated as
certified lower bounds (`PolicyGraph`), a solver that closes the gap between them at b0 (`GapSolver`) and exact value iteration with a
certified distance to V* (`IncrementalPruning_Solver`), none of them in the reference, backed by
hand-written sm_100a CUDA kernels in `libpbvi_b200.so` (C ABI: include/pbvi_b200.h).  The library is loaded on first
device use; without it (or without a CUDA device) the package raises -- there is no CPU fallback.
"""
from .model import Model, log  # noqa: F401

_LAZY = {
    'Belief': 'belief', 'BeliefSet': 'belief',
    'AlphaVector': 'value_function', 'ValueFunction': 'value_function',
    'PBVI_Solver': 'solver', 'HSVI_Solver': 'solver', 'FSVI_Solver': 'solver', 'FSVI_EG_Solver': 'solver',
    'VI_Solver': 'solver', 'BeliefValueMapping': 'solver', 'SolverHistory': 'solver', 'MDPSolverHistory': 'solver',
    'Agent': 'simulation', 'Simulation': 'simulation', 'SimulationSet': 'simulation', 'SimulationHistory': 'simulation',
    'RewardSet': 'simulation',
    'load_POMDP_file': 'pomdp_file', 'save_POMDP_file': 'pomdp_file', 'parse_POMDP': 'pomdp_file',
    'DeviceModel': '_native', 'ShardedBackup': 'parallel', 'ShardedSolveState': 'parallel', 'NativeComm': 'parallel',
    'FIB_Solver': 'bounds', 'UpperBound': 'bounds', 'PolicyGraph': 'policy_graph', 'ControllerOutcomes': 'policy_graph',
    'GapSolver': 'gap_solver', 'GapSolverHistory': 'gap_solver',
    'IncrementalPruning_Solver': 'incremental_pruning', 'IncrementalPruningHistory': 'incremental_pruning',
}


def __getattr__(name):
    # torch is imported only when a device-backed class is first touched (keeps `import` light for host-only tooling)
    if name in _LAZY:
        import importlib
        return getattr(importlib.import_module('.' + _LAZY[name], __name__), name)
    raise AttributeError(f'module {__name__!r} has no attribute {name!r}')
