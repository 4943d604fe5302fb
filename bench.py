#!/usr/bin/env python
"""
bench.py -- belief x alpha backups/sec of the PBVI backup on the olfactory-navigation POMDP (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--beliefs B] [--alphas V]
                    [--legs backup,solve,configs] [--scaling weak|strong] [--headline late|young|dense] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...          (one rank per GPU)

Workload (config.workload): BASELINE.json configs[2] -- the 22021-state toroidal olfactory model (A=6, O=3, R=1),
B = 10 000 belief points from Perseus random walks (100 walks x 100 steps from b0, the engine's own expand_perseus) backed up
against V = 1 000 alpha vectors.  One step = one full `PBVI_Solver.backup(model, belief_set, value_function)` pass = B*V
belief x alpha units: v* per (b,a,o), a*, assembly of the distinct alpha rows and the byte-dedup that forms the new alpha set.
Three value functions are measured, because the cost of a step depends on how much of the value function is exactly zero:

  late   (HEADLINE)  1 000 alphas produced by expansions >= 200 of the engine's own FSVI 300 x 100 solve of this model -- the
                     value function of a solve that has been running for a while (alpha density stated in the line);
  young              1 000 alphas grown by ~31 new-points backups from the initial value function (round-1 headline; 0.6 % dense);
  dense              the late alphas plus a strictly positive perturbation (no alpha-side zero at all).

At N > 1 every rank backs up its own B beliefs (weak scaling; `--scaling strong`: B beliefs in total, configs[3] uses 50 000) and
the ranks exchange + merge their generating tuples (pomdp_pbvi_exploration_b200.parallel).

`value`        device-resident inputs, CUDA-event timed, max over ranks.
`e2e`          the same call from HOST (pinned) buffers: H2D of beliefs and alphas, backup, D2H of the new alpha rows and actions.
`roofline`     the score kernel (block-sparse FP64 DMMA GEMM + fused argmax): EXECUTED flops / kernel time / FP64 tensor-pipe peak.
`parity_sample` the engine's v*, a* and alpha rows for a sample of the timed beliefs against the CPU oracle ON THE SAME ALPHAS, and the
               oracle's rows looked up bytewise in the output of the timed step.  A mismatch makes the run exit non-zero.
`cpu_baseline` the same oracle run (NumPy restatement of the reference's backup, oracle/pbvi_oracle.py), timed.
`solve`        whole solves (FSVI 300 x 100 as published by the reference; a full-backup Perseus solve with >= 10 000 beliefs), sharded
               over the ranks at N > 1 (`PBVI_Solver.solve(group=...)`).
`configs`      the other BASELINE configs (tiger, 4x4 grid, synthetic sparse sweep, sea-robin size), each with its own parity sample.
--impl reference runs the CPU oracle as the reference arm on the b200 arm's alphas.
--dump-outputs DIR writes the value function the last timed step of the headline point returned (dump_outputs()).  Every input is
generated from fixed seeds, so two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'belief x alpha backups/sec (olfactory POMDP S=22021, PBVI backup)'
UNIT = 'belief*alpha pairs/s'
GAMMA = 0.99
GAP_TOL = 1e-9                 # parity contract: indices identical wherever the oracle's top-2 gap exceeds GAP_TOL * max(1, |best|)
FP64_PEAK_TFLOPS = 37.1        # DMMA m8n8k4 / m16n8k16 on this pool's B200, profiles/r01_fp64_pipe_microbench.txt
# dram__bytes_read.sum + dram__bytes_write.sum of one score_kernel launch (`ncu --set full`, profiles/), per workload point at the
# default sizes (B = 10000, V = 1000); None = not captured
NCU_TRAFFIC_BYTES_PER_LAUNCH = {'young': 0.2400e9, 'late': 10.4627e9, 'dense': None}     # profiles/r02_score_kernel_{young,late}_ncu_summary.txt


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10,
                    help='timed steps of the value-function point the line reports; the other points run max(3, steps // 2), '
                         'the host-buffer leg runs steps')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--beliefs', type=int, default=10000, help='beliefs per GPU (weak scaling) or in total (--scaling strong)')
    ap.add_argument('--alphas', type=int, default=1000)
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'])
    ap.add_argument('--headline', default='late', choices=['late', 'young', 'dense'])
    ap.add_argument('--legs', default=None, help='comma list of backup,solve,configs (default: all three; at N > 1 the config leg runs a sharded subset)')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the oracle run (no parity_sample / cpu_baseline)')
    ap.add_argument('--parity-beliefs', type=int, default=None, help='beliefs of the oracle sample (default 512 at N = 1, 128 at N > 1)')
    ap.add_argument('--trace-phases', action='store_true', help='N > 1: print the phase times of the last sharded step to stderr')
    ap.add_argument('--no-e2e', action='store_true', help='skip the host-buffer leg (used for short ncu passes)')
    ap.add_argument('--only-point', default=None, help='measure one value-function point only (ncu passes)')
    ap.add_argument('--save-workload', default=None, help='write the synthetic beliefs / alphas to this .pt file')
    ap.add_argument('--load-workload', default=None, help='read them back instead of regenerating (ncu passes: no setup kernels)')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write the value function the last timed backup step returned to DIR/*.npy (float64, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or (args.legs and 'backup' not in args.legs.split(','))):
        ap.error('--dump-outputs needs the backup leg of --impl b200')
    return args


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """
    nvidia-smi clocks / throttle reasons, sampled every 100 ms from the warm-up on.  `begin()` / `end()` bracket the timed
    regions; the reported SM clock is the median of the samples that fall inside them (under load), or -- when a region is
    shorter than the sampling period -- of the samples of the 300 ms after it; throttle reasons come from the same samples.
    """
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []          # (arrival time, line)
        self.windows = []        # [begin, end] of the timed regions

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def begin(self):
        self.windows.append([time.perf_counter(), None])

    def end(self):
        if self.windows and self.windows[-1][1] is None:
            self.windows[-1][1] = time.perf_counter()

    def stop(self) -> dict:
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.3)
        self.proc.terminate()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        inside, after, mx, reasons = [], [], [], set()
        for t, ln in list(self.lines):
            parts = [p.strip() for p in ln.split(',')]
            if len(parts) < 7:
                continue
            try:
                clk, top = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            mx.append(top)
            if any(b <= t <= (e if e is not None else t) for b, e in self.windows):
                inside.append(clk)
            elif any(e is not None and e < t <= e + 0.3 for b, e in self.windows):
                after.append(clk)
            else:
                continue                                   # warm-up / set-up sample: neither its clock nor its reasons are reported
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        sm = inside if inside else after
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'samples': len(sm),
                'samples_total': len(mx), 'sampled': 'inside the timed regions' if inside else 'within 300 ms after a timed region',
                'reasons': sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------------
def use_all_host_threads() -> int:
    """The CPU arm uses every host core: torchrun exports OMP_NUM_THREADS=1 to its workers, which would leave NumPy's OpenBLAS (the
    reference's tensordot) single-threaded; threadpoolctl raises the limit at run time.  Returns the BLAS thread count in effect."""
    cores = os.cpu_count() or 1
    try:
        import torch
        torch.set_num_threads(cores)
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=cores)
        blas = [i['num_threads'] for i in threadpool_info() if i.get('user_api') == 'blas']
        return max(blas) if blas else cores
    except Exception:
        return cores


def seed_all(seed: int) -> None:
    np.random.seed(seed)
    random.seed(seed)


def timed_solve(solver, model, **kw):
    """A whole `solve` with wall clock (device-synchronised) and the time spent in compute_change; returns (vf, hist, summary dict)."""
    import torch
    change_s = [0.0]
    shard_change = [None]
    orig_change = solver.compute_change

    def timed_change(*a, **k):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = orig_change(*a, **k)
        torch.cuda.synchronize()
        change_s[0] += time.perf_counter() - t
        return out
    solver.compute_change = timed_change
    # units of a solve: every backup call processes (beliefs backed up) x (alphas of the value function it starts from)
    pair_count = [0.0]
    orig_backup = solver.backup

    def counted_backup(model_, belief_set, value_function, *a, **k):
        pair_count[0] += float(len(belief_set)) * len(value_function)
        return orig_backup(model_, belief_set, value_function, *a, **k)
    solver.backup = counted_backup
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vf, hist = solver.solve(model, print_progress=False, **kw)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    solver.compute_change, solver.backup = orig_change, orig_backup
    st = getattr(solver, '_shard_state', None)
    pairs = pair_count[0] + (st.stats.get('sharded_pairs', 0.0) if st is not None else 0.0)     # sharded backups: pairs of the WHOLE set
    out = dict(wall_s=wall, expand_s=float(sum(hist.expansion_times)), backup_s=float(sum(hist.backup_times)), change_s=change_s[0],
               expansions=len(hist.expansion_times), backups=len(hist.backup_times), final_alphas=len(vf), final_beliefs=int(hist.beliefs_counts[-1]),
               backup_pairs=pairs, backup_pairs_per_s=pairs / max(float(sum(hist.backup_times)), 1e-9))
    if st is not None:
        out['sharding'] = dict(st.stats)
    return vf, hist, out


def build_workload(model, n_beliefs: int, n_alphas: int, seed: int):
    """
    Synthetic inputs made by the engine itself.  Beliefs: Perseus walks (`seed`: per rank).  Value functions (the same on every rank):
    'young' grown by new-points backups from the initial one; 'late' taken from expansions >= 200 of an FSVI 300 x 100 solve.
    Returns (solver, beliefs, {'young': vf, 'late': vf}, info dict).
    """
    import torch
    from pomdp_pbvi_exploration_b200 import Belief, FSVI_Solver, PBVI_Solver, ValueFunction
    solver = PBVI_Solver(gamma=GAMMA, eps=1e-6, expand_function='perseus')
    np.random.seed(seed)
    walks = []
    b0 = Belief(model)
    n_walks = -(-n_beliefs // 100)
    for _ in range(n_walks):
        walks.append(solver.expand_perseus(model, b0, max_generation=100).belief_array)
    beliefs = torch.cat(walks)[:n_beliefs].contiguous()
    info = {}

    def pad_to(vf, rows, actions):
        if rows.shape[0] < n_alphas:                                # top up (not expected): perturbed copies keep the shape of the data
            g = torch.Generator(device='cpu').manual_seed(7)
            need = n_alphas - rows.shape[0]
            pick = torch.randint(0, rows.shape[0], (need,), generator=g)
            scale = 1.0 + 1e-3 * torch.rand((need, 1), generator=g, dtype=torch.float64)
            rows = torch.cat([rows, rows[pick.to(rows.device)] * scale.to(rows.device)])
            actions = np.concatenate([actions, actions[pick.numpy()]])
        return ValueFunction(model, rows[:n_alphas].contiguous(), actions[:n_alphas])

    # ---- young: FSVI/Perseus-style new-points backups over walks (append=True) until V >= n_alphas
    np.random.seed(1000)                                  # the alpha set is the same on every rank
    grow_walks = [solver.expand_perseus(model, b0, max_generation=100) for _ in range(40)]
    vf = ValueFunction(model, model.expected_rewards_table.T, model.actions)
    it = 0
    while len(vf) < n_alphas and it < 400:
        vf = solver.backup(model, grow_walks[it % len(grow_walks)], vf, append=True, belief_dominance_prune=False)
        it += 1
    young = pad_to(vf, vf.alpha_vector_array, vf.actions)
    info['young'] = {'provenance': f'{it} new-points backups over Perseus walks from the initial value function', 'growth_backups': it}

    # ---- late: the engine's own FSVI 300 x 100 solve (the reference's published shape); rows of expansions >= 200
    seed_all(0)
    FSVI_Solver(gamma=GAMMA, eps=1e-6).solve(model, expansions=3, max_belief_growth=100, print_progress=False)    # one-time costs (arena, module load)
    gpu_warm(model.device.device)
    seed_all(0)
    fsvi = FSVI_Solver(gamma=GAMMA, eps=1e-6)
    vf_f, hist, summary = timed_solve(fsvi, model, expansions=300, max_belief_growth=100)
    counts = hist.alpha_vector_counts                      # [initial, after backup 1, ...]
    cut = min(200, len(counts) - 1)
    n_late = len(vf_f) - counts[cut]                       # new rows are PREPENDED by every new-points backup: rows [0, n_late) are the late ones
    if n_late < n_alphas:
        n_late = min(len(vf_f), max(n_late, n_alphas))
    idx = np.unique(np.linspace(0, n_late - 1, min(n_alphas, n_late)).astype(np.int64))
    rows = vf_f.alpha_vector_array[torch.as_tensor(idx, device=vf_f.alpha_vector_array.device)]
    late = pad_to(vf_f, rows, vf_f.actions[idx])
    info['late'] = {'provenance': f'{len(idx)} alphas sampled evenly from the {n_late} rows that expansions >= {cut} of the engine\'s FSVI '
                                  f'300x100 solve (seed 0) produced; final |V| = {len(vf_f)}', 'fsvi_solve': summary}
    return solver, beliefs, {'young': young, 'late': late}, info


def make_dense(model, vf):
    import torch
    from pomdp_pbvi_exploration_b200 import ValueFunction
    g = torch.Generator(device='cpu').manual_seed(11)
    noise = (1e-3 * torch.rand(vf.alpha_vector_array.shape, generator=g, dtype=torch.float64) + 1e-6).to(vf.alpha_vector_array.device)
    return ValueFunction(model, vf.alpha_vector_array + noise, vf.actions)


# ---------------------------------------------------------------------------------------------------------------------
def oracle_backup_sample(reach, rto, rbar, gamma, beliefs_host: np.ndarray, alphas_host: np.ndarray, chunk: int = 512):
    """
    The reference's backup arithmetic (NumPy restatement, oracle/pbvi_oracle.py: same primitives, same order as src/pomdp.py:1485-1506)
    on `beliefs_host`, in chunks of `chunk` rows (BASELINE.md section 3: the reference itself needs belief chunks at this size: Gamma* is
    8*B*A*O*S bytes).  Returns (outputs dict, timing dict): the Gamma projection is timed separately because its cost does not depend
    on the number of beliefs.
    """
    from oracle import pbvi_oracle as orc
    A, O, S = rto.shape[1], rto.shape[2], rto.shape[0]
    t0 = time.perf_counter()
    G = orc.gamma_projection(reach, rto, alphas_host, gamma)
    t_gamma = time.perf_counter() - t0
    outs = {k: [] for k in ('v_star', 'a_star', 'alpha', 'values', 'best', 'gap')}
    t0 = time.perf_counter()
    t_extra = 0.0
    for i0 in range(0, beliefs_host.shape[0], chunk):
        b = beliefs_host[i0:i0 + chunk]
        scores = np.tensordot(b, G, (1, 3))
        v_star = np.argmax(scores, axis=3)
        best_per_o = G[np.arange(A)[None, :, None, None], np.arange(O)[None, None, :, None], v_star[:, :, :, None], np.arange(S)[None, None, None, :]]
        alpha_a = rbar.T + np.sum(best_per_o, axis=2)
        values = np.einsum('bas,bs->ba', alpha_a, b)
        a_star = np.argmax(values, axis=1)
        rows = np.take_along_axis(alpha_a, a_star[:, None, None], axis=1)[:, 0, :]
        orc.dedup_rows(rows, a_star)
        te = time.perf_counter()                      # (not part of the reference's work: top-2 gaps for the parity contract)
        if scores.shape[3] > 1:
            top = np.partition(scores, scores.shape[3] - 2, axis=3)[..., -2:]
            outs['best'].append(top[..., 1]); outs['gap'].append(top[..., 1] - top[..., 0])
        else:
            outs['best'].append(scores[..., 0]); outs['gap'].append(np.full(scores.shape[:3], np.inf))
        for k, v in (('v_star', v_star), ('a_star', a_star), ('alpha', rows), ('values', values)):
            outs[k].append(v)
        t_extra += time.perf_counter() - te
    t_rows = time.perf_counter() - t0 - t_extra
    out = {k: np.concatenate(v) for k, v in outs.items()}
    return out, {'gamma_projection_s': t_gamma, 'per_belief_part_s': t_rows, 'sample_beliefs': int(beliefs_host.shape[0]), 'chunk_rows': chunk}


def extrapolate(timing: dict, n_full: int, n_alphas: int) -> dict:
    """pairs/s of the full step from a timed sample: Gamma projection once + the per-belief part scaled linearly in B."""
    n = timing['sample_beliefs']
    t_full = timing['gamma_projection_s'] + timing['per_belief_part_s'] * (n_full / n)
    t_sample = timing['gamma_projection_s'] + timing['per_belief_part_s']
    return {'value': n_full * n_alphas / t_full, 'full_step_s_estimate': t_full, 'extrapolation_factor': n_full / n,
            'sample_pairs_per_s_raw': n * n_alphas / t_sample, 'sample_s': t_sample}


def parity_check(dev, host_model, gamma, sample_beliefs, vf, ref: dict, step_output=None) -> dict:
    """
    The engine (through the C ABI, `DeviceModel.backup`: select + assemble for every belief) against the oracle outputs `ref` on the same
    beliefs and alphas.  Contract: v* / a* identical wherever the oracle's top-2 gap is decided; rows bit-identical where both chose the
    same tuple (R = 1) / within 1e-9 (R > 1).  With `step_output` (the ValueFunction the timed step returned) every oracle row of a
    decided belief must also occur, bytewise, in that output.
    """
    import torch
    reach = host_model['reach']
    alpha, act, vstar, value = [t.cpu().numpy() for t in dev.backup(sample_beliefs, vf.alpha_vector_array, gamma)]
    scale = np.maximum(1.0, np.abs(ref['best']))
    decided = ref['gap'] > GAP_TOL * scale
    v_bad = int(np.sum(vstar[decided] != ref['v_star'][decided]))
    vs = np.sort(ref['values'], axis=1)
    agap = vs[:, -1] - vs[:, -2] if vs.shape[1] > 1 else np.full(vs.shape[0], np.inf)
    adecided = agap > GAP_TOL * np.maximum(1.0, np.abs(vs[:, -1]))
    a_bad = int(np.sum(act[adecided] != ref['a_star'][adecided]))
    ours_sel = np.take_along_axis(vstar, act[:, None, None].astype(np.int64), axis=1)[:, 0, :]
    ref_sel = np.take_along_axis(ref['v_star'], ref['a_star'][:, None, None], axis=1)[:, 0, :]
    same = (act == ref['a_star']) & np.all(ours_sel == ref_sel, axis=1)
    exact = reach.shape[2] == 1
    if exact:
        rows_equal = int(np.sum(np.all(alpha[same].view(np.uint64) == ref['alpha'][same].view(np.uint64), axis=1)))
        max_rel = 0.0 if rows_equal == int(same.sum()) else float(np.max(np.abs(alpha[same] - ref['alpha'][same])))
    else:
        close = np.isclose(alpha[same], ref['alpha'][same], rtol=1e-9, atol=1e-12).all(axis=1)
        rows_equal = int(close.sum())
        max_rel = float(np.max(np.abs(alpha[same] - ref['alpha'][same]) / np.maximum(1e-300, np.abs(ref['alpha'][same])))) if same.any() else 0.0
    out = {'beliefs': int(sample_beliefs.shape[0]), 'alphas': int(len(vf)), 'vstar_compared_decided': int(decided.sum()),
           'vstar_mismatch_decided': v_bad, 'astar_compared_decided': int(adecided.sum()), 'astar_mismatch_decided': a_bad,
           'rows_compared': int(same.sum()), 'rows_bitwise_equal' if exact else 'rows_within_1e-9': rows_equal, 'max_abs_row_diff': max_rel,
           'gap_tolerance': GAP_TOL}
    ok = v_bad == 0 and a_bad == 0 and rows_equal == int(same.sum())
    if step_output is not None and exact:
        # the oracle's rows of the decided beliefs must be rows of the timed step's value function: 128-bit keys, then bytes
        want = ref['alpha'][same & adecided]
        keys_out = step_output.row_hashes
        index = {tuple(k): i for i, k in enumerate(keys_out.tolist())}
        d_want = torch.as_tensor(want).to(dev.device)
        keys_want = dev.row_hash(d_want).cpu().numpy().tolist()
        pos = [index.get(tuple(k), -1) for k in keys_want]
        found = [i for i, p in enumerate(pos) if p >= 0]
        n_found = 0
        if found:
            flags = dev.rows_equal(d_want, np.array(found, dtype=np.int32), step_output.alpha_vector_array, np.array([pos[i] for i in found], dtype=np.int32))
            n_found = int(flags.sum())
        out['oracle_rows_looked_up_in_step_output'] = int(want.shape[0])
        out['oracle_rows_found_bytewise_in_step_output'] = n_found
        ok = ok and n_found == int(want.shape[0])
    out['ok'] = bool(ok)
    return out


def host_tables(model) -> dict:
    return {'reach': model.reachable_states, 'rto': model.reachable_transitional_observation_table, 'rbar': model.expected_rewards_table}


def dump_outputs(directory: str, vf, max_bytes: int = 64 << 20) -> dict:
    """
    Writes the ValueFunction a timed backup step returned, as float64 .npy files, so that two builds run with the same arguments can
    be compared output for output:
      actions.npy                      the action of every new alpha row;
      alpha_vector_row_sums.npy        the sum over states of every new alpha row;
      alpha_vector_array.npy           the rows themselves -- all of them, or, when they do not fit in `max_bytes` with the two
                                       arrays above, a sample drawn with a fixed seed (sorted);
      alpha_vector_array_rows.npy      the positions of those rows in the value function.
    """
    import torch
    rows = vf.alpha_vector_array                         # summed and sampled where it lives: only the sampled rows are copied back
    n, S = rows.shape
    fit = max(0, (max_bytes - 4096 - 2 * n * 8) // ((S + 1) * 8))          # (4096: the four .npy headers)
    pick = np.arange(n) if fit >= n else np.sort(np.random.default_rng(0).choice(n, fit, replace=False))
    arrays = {'actions': np.asarray(vf.actions, dtype=np.float64), 'alpha_vector_row_sums': rows.sum(dim=1).cpu().numpy(),
              'alpha_vector_array': rows[torch.as_tensor(pick, device=rows.device)].cpu().numpy(),
              'alpha_vector_array_rows': pick.astype(np.float64)}
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + '.npy'), a)
    return {'dir': directory, 'alpha_rows': n, 'alpha_rows_written': int(pick.size),
            'bytes': int(sum(a.nbytes for a in arrays.values()))}


# ---------------------------------------------------------------------------------------------------------------------
def workload_config(args, world, headline=None, density=None):
    per_gpu = args.beliefs if args.scaling == 'weak' else -(-args.beliefs // world)
    cfg = {'workload': f'olfactory_wrap S=22021 A=6 O=3 R=1 (BASELINE configs[2]): Perseus-walk beliefs B={per_gpu}/GPU x V={args.alphas} alphas, '
                       f'full PBVI backup incl. dedup; value function: {headline or args.headline}',
           'beliefs_per_gpu': per_gpu, 'beliefs_total': per_gpu * world, 'alphas': args.alphas, 'gamma': GAMMA,
           'value_function': headline or args.headline,
           'parallelism': f'belief-sharded x{world}' if world > 1 else 'single GPU',
           'l2_policy': 'inputs larger than L2 (beliefs 1.76 GB, alphaT 0.18 GB per step)'}
    if density:
        cfg.update(density)
    return cfg


def run_reference(args):
    """
    Reference arm: the reference's CPU algorithm (oracle port; the Python reference itself cannot travel to the GPU box) on the b200
    arm's workload.  The value function is the b200 arm's (built by the engine when a GPU is present -- that construction is not
    timed and nothing of the engine runs inside the timed region), each step = the whole backup arithmetic on a bounded sample of
    the B beliefs in 512-row chunks; `value` extrapolates linearly in B to the full step (factor printed).
    """
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if rank != 0:
        return
    import torch
    from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model, perseus_walk_beliefs
    model = olfactory_wrap_model()
    cores = use_all_host_threads()
    n_full = (args.beliefs if args.scaling == 'weak' else -(-args.beliefs // world)) * world
    n_sample = min(n_full, 512 if args.steps + args.warmup <= 16 else 256)
    built_by = 'numpy (no CUDA device): Rbar rows + smooth random rows'
    density = None
    if torch.cuda.is_available():
        try:
            torch.cuda.set_device(0)
            _, beliefs_d, vfs, info = build_workload(model, n_sample, args.alphas, seed=0)
            vf = vfs[args.headline] if args.headline != 'dense' else make_dense(model, vfs['late'])
            alphas = vf.alpha_vector_array.cpu().numpy()
            beliefs = beliefs_d.cpu().numpy()
            density = {'alpha_density': float((alphas != 0).mean()), 'belief_density': float((beliefs != 0).mean())}
            built_by = f'the b200 engine, untimed ({info.get(args.headline, info["late"])["provenance"]})'
            model.device.close()
            torch.cuda.empty_cache()
        except Exception as e:                     # the reference arm must not depend on the engine
            print(f'[reference arm] engine-built workload unavailable ({e}); using the numpy stand-in', file=sys.stderr)
            beliefs = None
    else:
        beliefs = None
    if beliefs is None:
        beliefs = perseus_walk_beliefs(model, n_sample, seed=0)
        rng = np.random.default_rng(0)
        alphas = np.concatenate([model.expected_rewards_table.T, rng.random((args.alphas - model.action_count, model.state_count)) * 0.1])
    tabs = host_tables(model)
    vals = []
    for step in range(args.warmup + args.steps):
        _, timing = oracle_backup_sample(tabs['reach'], tabs['rto'], tabs['rbar'], GAMMA, beliefs, alphas, chunk=512)
        if step >= args.warmup:
            vals.append((extrapolate(timing, n_full, args.alphas), timing))
    value = float(np.mean([v['value'] for v, _ in vals]))
    ext, timing = vals[-1]
    sample = (f'per step: Gamma projection for all {args.alphas} alphas + per-belief part on {n_sample} of {n_full} beliefs in 512-row chunks, '
              f'extrapolated linearly in B (factor {n_full / n_sample:.1f}); NumPy/OpenBLAS, {cores} threads; alphas built by {built_by}')
    emit(({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': float(np.mean([v['sample_s'] for v, _ in vals])) * 1e3, 'higher_is_better': True, 'scaling': args.scaling,
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(args, world, density=density),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample,
                         'ms_per_step_is': 'the measured time of one SAMPLE step', **{k: v for k, v in ext.items() if k != 'value'}, **timing},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


# ---------------------------------------------------------------------------------------------------------------------
def gpu_warm(device, seconds: float = 0.4) -> None:
    """Keeps the GPU busy for a moment (plain torch matmuls): after seconds of idling behind a CPU-only phase the SM clocks are down, and
    a launch-bound leg measured right then would be timed at idle clocks."""
    import torch
    a = torch.rand((2048, 2048), device=device)
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        for _ in range(20):
            a = (a @ a).clamp_(0, 1)
        torch.cuda.synchronize(device)


def time_device_steps(step_fn, dev, steps, warmup, barrier, sampler):
    import torch
    for _ in range(warmup):
        out = step_fn()
    dev.set_profiling(True)
    barrier()
    launches0 = dev.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    score_ms = []
    sampler.begin()
    ev0.record()
    for _ in range(steps):
        out = step_fn()
        score_ms.append(dev.last_score_ms())       # the step has already synchronised (dedup reads counts back)
    ev1.record()
    barrier()
    sampler.end()
    stats = dev.last_stats()
    return {'out': out, 'elapsed_ms': ev0.elapsed_time(ev1), 'score_ms': float(np.mean(score_ms)), 'launches': dev.launch_count - launches0,
            'executed_flops': stats['executed_flops'], 'dense_flops': stats['dense_flops']}


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from pomdp_pbvi_exploration_b200 import BeliefSet, PBVI_Solver, ValueFunction
    from pomdp_pbvi_exploration_b200.parallel import ShardedBackup
    from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model

    legs = args.legs.split(',') if args.legs else ['backup', 'solve', 'configs']
    model = olfactory_wrap_model()
    dev = model.device
    per_gpu = args.beliefs if args.scaling == 'weak' else -(-args.beliefs // world)
    info = {}
    if args.load_workload:
        blob = torch.load(args.load_workload)
        solver = PBVI_Solver(gamma=GAMMA, eps=1e-6, expand_function='perseus')
        beliefs = blob['beliefs'].to(dev.device)
        vfs = {k: ValueFunction(model, blob[k + '_alphas'].to(dev.device), blob[k + '_actions'].numpy()) for k in ('young', 'late')}
        info = blob['info']
    else:
        solver, beliefs, vfs, info = build_workload(model, per_gpu, args.alphas, seed=rank)
    if args.save_workload and rank == 0:
        torch.save({'beliefs': beliefs.cpu(), 'info': info,
                    **{k + '_alphas': v.alpha_vector_array.cpu() for k, v in vfs.items()}, **{k + '_actions': torch.as_tensor(v.actions) for k, v in vfs.items()}},
                   args.save_workload)
    vfs['dense'] = make_dense(model, vfs['late'])
    info['dense'] = {'provenance': 'the late alphas plus a strictly positive perturbation (every alpha non-zero at every state)'}
    B, V = beliefs.shape[0], len(vfs[args.headline])
    A, O, S = model.action_count, model.observation_count, model.state_count
    belief_set = BeliefSet(model, beliefs)
    sharded = ShardedBackup(solver, model) if world > 1 else None
    if sharded is not None:
        sharded.set_capacity(B)            # every rank backs up exactly B beliefs

    def make_step(vf):
        def step():
            if sharded is not None:
                return sharded.backup(belief_set, vf, append=False)
            return solver.backup(model, belief_set, vf, append=False, belief_dominance_prune=False)
        return step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(vals, dtype=torch.float64, device=dev.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    line = None
    results = {}
    belief_density = float((beliefs != 0).double().mean())
    if 'backup' in legs:
        # ---- device-resident timing: the headline value function first, then the other two points --------------------
        sampler = ClockSampler(local_rank)
        sampler.start()                     # started before the warm-up so that nvidia-smi is up when the timed regions run
        order = [args.headline] + [k for k in ('late', 'young', 'dense') if k != args.headline]
        if args.only_point:
            order = [args.only_point]
        for name in order:
            n_steps = args.steps if name == order[0] else max(3, args.steps // 2)        # order[0]: the point the line reports
            n_warm = args.warmup if name == order[0] else max(2, args.warmup // 2)
            r = time_device_steps(make_step(vfs[name]), dev, n_steps, n_warm, barrier, sampler)
            r['steps'] = n_steps
            r['elapsed_ms'], r['score_ms'] = reduce_max([r['elapsed_ms'], r['score_ms']])
            r['alpha_density'] = float((vfs[name].alpha_vector_array != 0).double().mean())
            results[name] = r
        if args.trace_phases and sharded is not None:
            sharded.trace = True
            make_step(vfs[args.headline])()
            sharded.trace = False
            print(f'[rank {rank}] phases (ms): ' + json.dumps({k: round(v, 3) for k, v in sharded.last_phases.items()}), file=sys.stderr)
        clocks = sampler.stop()       # before the e2e leg: that one is PCIe-bound, the GPU idles through part of it
        head = results[order[0]]
        vf_head = vfs[order[0]]
        out = head['out']

        # ---- end to end from host buffers -----------------------------------------------------------------------------
        h_beliefs = beliefs.cpu().pin_memory()
        h_alphas = vf_head.alpha_vector_array.cpu().pin_memory()
        h_actions = vf_head.actions.copy()

        def step_e2e():
            bs = BeliefSet(model, h_beliefs)                             # H2D
            v_in = ValueFunction(model, h_alphas, h_actions)            # H2D (+ the constructor's byte-dedup)
            if sharded is not None:
                res = sharded.backup(bs, v_in, append=False)
            else:
                res = solver.backup(model, bs, v_in, append=False, belief_dominance_prune=False)
            return res.numpy(staged=True)                                # D2H into the pinned staging buffer

        e2e_steps = 0 if args.no_e2e else args.steps
        for _ in range(0 if args.no_e2e else args.warmup):
            rows, acts = step_e2e()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rows, acts = np.zeros((0, S)), np.zeros(0)
        for _ in range(e2e_steps):
            rows, acts = step_e2e()
        e1.record()
        barrier()
        e2e_ms = e0.elapsed_time(e1) if e2e_steps else 0.0   # device clock; every step ends with the blocking D2H read
        # bytes that actually crossed PCIe per step: the belief rows travel packed (bitmap + non-zero 4-double chunks, packed by host
        # threads inside the timed region and rebuilt bytewise on the device), the alpha rows as they are
        h2d_dense = int(h_beliefs.numel() * 8 + h_alphas.numel() * 8)
        h2d = int(getattr(solver, 'last_h2d_bytes', h_beliefs.numel() * 8) + h_alphas.numel() * 8) if e2e_steps else h2d_dense
        d2h = int(rows.size * 8 + acts.size * 8)
        (e2e_ms,) = reduce_max([e2e_ms])
        # the same backup through the C ABI alone (what a non-Python host binds, INTEGRATION.md): one pbvi_backup_host_unique call,
        # from page-locked buffers and from plain (pageable) NumPy arrays; its rows must be the step's rows
        c_abi = None
        if e2e_steps and world == 1:
            import ctypes
            n_out = ctypes.c_int()
            cap = int(min(B, 4 * rows.shape[0] + 64))
            st = torch.cuda.current_stream().cuda_stream
            o_rows, o_act = torch.empty((cap, S), dtype=torch.float64).pin_memory(), torch.empty((cap,), dtype=torch.int32).pin_memory()
            p_b, p_a = h_beliefs.numpy().copy(), h_alphas.numpy().copy()
            p_rows, p_act = np.empty((cap, S)), np.empty(cap, dtype=np.int32)

            def call(b_ptr, a_ptr, r_ptr, act_ptr):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rc = dev._lib.pbvi_backup_host_unique(dev._h, b_ptr, B, a_ptr, V, ctypes.c_double(GAMMA), r_ptr, cap, act_ptr, ctypes.byref(n_out), st)
                assert rc == 0, dev._lib.pbvi_last_error()
                return (time.perf_counter() - t0) * 1e3
            pinned_ms = [call(h_beliefs.data_ptr(), h_alphas.data_ptr(), o_rows.data_ptr(), o_act.data_ptr()) for _ in range(5)][2:]
            pageable_ms = [call(p_b.ctypes.data, p_a.ctypes.data, p_rows.ctypes.data, p_act.ctypes.data) for _ in range(5)][2:]
            c_abi = {'entry': 'pbvi_backup_host_unique (whole backup incl. the ValueFunction-constructor dedup, host buffers in and out)',
                     'ms_per_call_pinned': float(np.mean(pinned_ms)), 'ms_per_call_pageable_numpy': float(np.mean(pageable_ms)),
                     'rows': int(n_out.value),
                     'rows_equal_step_output': bool(n_out.value == rows.shape[0] and np.array_equal(p_rows[:n_out.value], rows)
                                                    and np.array_equal(o_rows[:n_out.value].numpy(), rows)
                                                    and np.array_equal(p_act[:n_out.value], np.asarray(acts)))}

        units = float(B) * V * world
        ms_step = head['elapsed_ms'] / head['steps']
        algo_flops = 2.0 * A * O * S * B * V                  # per launch (per rank), dense count
        exec_tflops = head['executed_flops'] / (head['score_ms'] * 1e-3) / 1e12
        points = {}
        for name, r in results.items():
            ms = r['elapsed_ms'] / r['steps']
            points[name] = {'value': float(B) * len(vfs[name]) * world / (ms * 1e-3), 'ms_per_step': ms, 'kernel_ms': r['score_ms'],
                            'alpha_density': r['alpha_density'], 'executed_flops_per_launch': r['executed_flops'],
                            'executed_over_algorithmic': r['executed_flops'] / algo_flops,
                            'executed_tflops': r['executed_flops'] / (r['score_ms'] * 1e-3) / 1e12,
                            'pipe_frac': r['executed_flops'] / (r['score_ms'] * 1e-3) / 1e12 / FP64_PEAK_TFLOPS,
                            'new_alpha_rows': len(r['out']), 'provenance': info.get(name, {}).get('provenance')}
        line = {
            'metric': METRIC, 'value': units / (ms_step * 1e-3), 'unit': UNIT, 'n_gpus': world, 'steps': head['steps'], 'warmup': args.warmup,
            'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f64',
            'data': 'synthetic',
            'config': workload_config(args, world, order[0], {'alpha_density': head['alpha_density'], 'belief_density': belief_density,
                                                               'value_function_provenance': info.get(order[0], {}).get('provenance')}),
            'clocks': clocks,
            'e2e': {'value': units * args.steps / (e2e_ms * 1e-3) if e2e_ms > 0 else None, 'unit': UNIT, 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h, 'ms_per_step': (e2e_ms / args.steps) if e2e_ms > 0 else None,
                    'c_abi': c_abi, 'host_input_bytes_per_step': h2d_dense, 'host_threads': (dev.__dict__.get('_pack') or {}).get('pool')._max_workers if (e2e_steps and h2d < h2d_dense) else 1,
                    'api': 'BeliefSet(host) + ValueFunction(host) -> PBVI_Solver.backup -> ValueFunction.numpy(); sparse belief rows are packed by '
                           'host threads (pbvi_pack_slabs_host) for the upload and unpacked on the device; the alpha rows known before the last '
                           'chunk of beliefs is scored are read back beside that kernel'},
            'gpu_launches': int(head['launches']),
            'roofline': {'bound': 'tensor', 'kernel': 'score_kernel<GATHER> (persistent block-sparse FP64 DMMA m8n8k4 GEMM + fused argmax)',
                         'achieved': exec_tflops, 'peak': FP64_PEAK_TFLOPS, 'unit': 'TFLOP/s', 'frac': exec_tflops / FP64_PEAK_TFLOPS,
                         'traffic': NCU_TRAFFIC_BYTES_PER_LAUNCH.get(order[0]) if (B == 10000 and V == 1000) else None,
                         'peak_source': 'own FP64 DMMA microbenchmark on this pool (profiles/r01_fp64_pipe_microbench.txt); '
                                        'MEASURED_PEAKS.json has no FP64 entry (cuBLAS DGEMM reaches 35.5 on the same box)',
                         'flops_counted': 'EXECUTED flops of the launch (2 * 16 beliefs * 64 alphas * 4 states per visited (chunk, row group, '
                                          'column quarter), counted by the kernel); skipped terms are exact zeros',
                         'executed_flops_per_launch': head['executed_flops'], 'algorithmic_flops_per_launch': algo_flops,
                         'algorithmic_over_executed': algo_flops / max(head['executed_flops'], 1.0),
                         'kernel_ms': head['score_ms'], 'kernel_share_of_step': head['score_ms'] / ms_step},
            'value_function_points': points,
        }

    # ---- whole solves ---------------------------------------------------------------------------------------------------------
    if 'solve' in legs:
        # (before the CPU oracle leg: several seconds of an idle GPU let its clocks drop, and a launch-bound solve that starts right
        # after that runs several times slower until they are back up)
        solve = {}
        gpu_warm(dev.device)
        try:
            solve = run_solve_leg(model, world, rank, info, reduce_max)
        except Exception as e:          # the solve leg must not take the headline down with it
            solve = {'error': f'{type(e).__name__}: {e}'}
        if line is not None:
            line['solve'] = solve
        elif rank == 0:
            line = {'metric': 'PBVI solve wall time', 'solve': solve, 'n_gpus': world}
    # ---- parity sample + CPU baseline: the oracle on the headline alphas, for a sample of the timed beliefs (rank 0) -----------------
    parity_failed = False
    if 'backup' in legs and rank == 0 and not args.no_cpu_baseline:
        prev_threads = torch.get_num_threads()
        cores = use_all_host_threads()
        n_sample = min(B, args.parity_beliefs or (512 if world == 1 else 128))
        pick = np.unique(np.linspace(0, B - 1, n_sample).astype(np.int64))
        sample_b = beliefs[torch.as_tensor(pick, device=dev.device)]
        tabs = host_tables(model)
        ref, timing = oracle_backup_sample(tabs['reach'], tabs['rto'], tabs['rbar'], GAMMA, sample_b.cpu().numpy(),
                                           vf_head.alpha_vector_array.cpu().numpy(), chunk=512)
        line['parity_sample'] = parity_check(dev, tabs, GAMMA, sample_b, vf_head, ref, step_output=out)
        line['parity_sample']['what'] = (f'{len(pick)} of the {B} timed beliefs (evenly spaced), the headline value function; oracle = '
                                         'oracle/pbvi_oracle.py (NumPy restatement of src/pomdp.py:1485-1506)')
        parity_failed = not line['parity_sample']['ok']
        if world == 1:
            ext = extrapolate(timing, B, V)
            line['cpu_baseline'] = {'value': ext['value'], 'unit': UNIT, 'cores': cores, 'kind': 'port',
                                    'sample': f'Gamma projection for all {V} alphas + per-belief part on {len(pick)} of {B} beliefs in 512-row chunks, '
                                              f'extrapolated linearly in B (factor {ext["extrapolation_factor"]:.1f}); NumPy/OpenBLAS with {cores} threads; '
                                              'the same alphas and beliefs as the timed step',
                                    **{k: v for k, v in ext.items() if k != 'value'}, **timing}
        torch.set_num_threads(prev_threads)

    if 'solve' in legs and rank == 0 and line is not None and 'cpu_baseline' in line and 'error' not in line.get('solve', {'error': 1}):
        solve = line['solve']
        if True:
            cpu = line['cpu_baseline']['value']
            for k, s in solve.items():
                if isinstance(s, dict) and 'backup_pairs' in s:
                    s['cpu_port_backup_s_estimate'] = s['backup_pairs'] / cpu
                    s['cpu_port_estimate_note'] = ('backup pairs of this solve / the cpu_baseline pairs-per-second of this run (late value '
                                                   'function, B = 10 000): an estimate of the reference CPU path\'s backup time alone')

    if 'configs' in legs and world == 1 and rank == 0:
        gpu_warm(dev.device)
        try:
            line['configs'] = run_config_leg(args)
        except Exception as e:
            line['configs'] = {'error': f'{type(e).__name__}: {e}'}
    elif 'configs' in legs and world > 1:
        gpu_warm(dev.device)
        cfg = run_config_leg_sharded(world, rank)          # every rank takes part (collectives); rank 0 keeps the records
        if rank == 0 and line is not None:
            line['configs'] = cfg

    if args.dump_outputs and rank == 0:                   # (parse_args: the backup leg ran, `out` is its headline step's output)
        line['dump_outputs'] = dump_outputs(args.dump_outputs, out)
    if rank == 0 and line is not None:
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    if parity_failed:
        sys.exit(3)


def run_solve_leg(model, world, rank, info, reduce_max) -> dict:
    """
    Whole solves of the olfactory model, device-synchronised wall clock, max over ranks:
      fsvi_300x100           the reference's published shape (2983.5 s NumPy CPU, 204.9 s CuPy GPU: BASELINE.md section 1);
      perseus_full_10k       PBVI_Solver('perseus').solve(expansions=2, max_belief_growth=6000, full_backup=True, update_passes=15):
                             the Perseus scheme -- a belief set collected by random walks (12 000 walk steps; > 10 000 distinct beliefs,
                             north_star: ">= 10k belief points"), then repeated backups of the WHOLE set (`update_passes` is the
                             reference's own parameter, src/pomdp.py:2172-2186), each followed by compute_change.
      pbvi_full_backup_fsvi_200x100  classic PBVI: PBVI_Solver('fsvi').solve(expansions=200, max_belief_growth=100, full_backup=True) -- FSVI
                             exploration, but EVERY expansion backs up the whole belief set (8 437 beliefs at the end, 2.5e9 pairs): the
                             solve whose time is in the phases that shard.
    At N > 1 the loop is sharded over the ranks (`solve(group=True)`).
    """
    from pomdp_pbvi_exploration_b200 import FSVI_Solver, PBVI_Solver
    out = {}
    shard = {'group': True} if world > 1 else {}
    if world == 1 and 'late' in info and 'fsvi_solve' in info['late']:
        # the solve that produced the workload ran with a cold scratch arena (it grows with |V|); the same solve again, like at N > 1
        out['fsvi_300x100_first_run_in_process'] = dict(info['late']['fsvi_solve'])
    gpu_warm(model.device.device)
    seed_all(0)
    _, _, s = timed_solve(FSVI_Solver(gamma=GAMMA, eps=1e-6), model, expansions=300, max_belief_growth=100, **shard)
    s['wall_s'], s['expand_s'], s['backup_s'], s['change_s'] = reduce_max([s['wall_s'], s['expand_s'], s['backup_s'], s['change_s']])
    s['reference_published'] = {'numpy_cpu_s': 2983.5, 'cupy_gpu_s': 204.9, 'source': 'Olfactory_Alternation_Paper_Wrap.ipynb[43],[30] (BASELINE.md)'}
    out['fsvi_300x100'] = s
    gpu_warm(model.device.device)
    seed_all(0)
    _, _, s = timed_solve(PBVI_Solver(gamma=GAMMA, eps=1e-6, expand_function='perseus'), model, expansions=2, max_belief_growth=6000,
                          full_backup=True, update_passes=15, **shard)
    s['wall_s'], s['expand_s'], s['backup_s'], s['change_s'] = reduce_max([s['wall_s'], s['expand_s'], s['backup_s'], s['change_s']])
    out['perseus_full_10k'] = s
    gpu_warm(model.device.device)
    seed_all(0)
    _, _, s = timed_solve(PBVI_Solver(gamma=GAMMA, eps=1e-6, expand_function='fsvi'), model, expansions=200, max_belief_growth=100,
                          full_backup=True, **shard)
    s['wall_s'], s['expand_s'], s['backup_s'], s['change_s'] = reduce_max([s['wall_s'], s['expand_s'], s['backup_s'], s['change_s']])
    out['pbvi_full_backup_fsvi_200x100'] = s
    out['n_gpus'] = world
    out['note'] = ('expansions draw on the host RNG and are sequential in the belief (b_{t+1} depends on o_t): they run on rank 0 and are '
                   'broadcast; backups and compute_change are sharded')
    return out


# ---------------------------------------------------------------------------------------------------------------------
def _time_backup(model, gamma, B, V, acts, reps, world=1):
    """ms per `PBVI_Solver.backup` of the belief set B (CUDA events).  world > 1: the SAME belief set sharded over the ranks (strong
    scaling: contiguous row blocks, tuple exchange), time = max over ranks."""
    import torch
    from pomdp_pbvi_exploration_b200 import BeliefSet, PBVI_Solver, ValueFunction
    solver = PBVI_Solver(gamma=gamma, eps=1e-6, expand_function='ssea')
    vf = ValueFunction(model, V, acts)
    if world > 1:
        import torch.distributed as dist
        from pomdp_pbvi_exploration_b200.parallel import ShardedBackup
        sb = ShardedBackup(solver, model)
        lo, hi = sb.bounds(B.shape[0])
        bs = BeliefSet(model, np.ascontiguousarray(B[lo:hi]) if hi > lo else torch.empty((0, B.shape[1]), dtype=torch.float64, device=model.device.device))
        step = lambda: sb.backup(bs, vf, append=False)
    else:
        bs = BeliefSet(model, B)
        step = lambda: solver.backup(model, bs, vf, append=False, belief_dominance_prune=False)
    for _ in range(3):
        out = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=model.device.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
    return ms, out, vf


def _dirichlet_beliefs(rng, n, S, k):
    B = np.zeros((n, S))
    for i in range(n):
        idx = rng.choice(S, min(k, S), replace=False)
        B[i, idx] = rng.dirichlet(np.ones(len(idx)))
    return B


def _config_point(name, model, gamma, B, V, acts, reps, parity_rows, world=1, rank=0):
    """One backup shape of another model: time per backup (CUDA events), pairs/s, and a parity sample against the oracle."""
    import torch
    ms, out, vf = _time_backup(model, gamma, B, V, acts, reps, world)
    if rank != 0:
        return None
    S, A, O, R = model.state_count, model.action_count, model.observation_count, model.reachable_state_count
    rec = {'config': name, 'S': S, 'A': A, 'O': O, 'R': R, 'B': int(B.shape[0]), 'V': len(vf), 'ms_per_backup': ms,
           'pairs_per_s': B.shape[0] * len(vf) / (ms * 1e-3), 'new_alpha_rows': len(out),
           'algorithmic_tflops': 2.0 * A * O * S * B.shape[0] * len(vf) / (ms * 1e-3) / 1e12}
    if parity_rows:
        tabs = host_tables(model)
        pick = np.unique(np.linspace(0, B.shape[0] - 1, min(parity_rows, B.shape[0])).astype(np.int64))
        sb = np.ascontiguousarray(B[pick])
        t0 = time.perf_counter()
        ref, timing = oracle_backup_sample(tabs['reach'], tabs['rto'], tabs['rbar'], gamma, sb, vf.alpha_vector_array.cpu().numpy(), chunk=256)
        rec['parity_sample'] = parity_check(model.device, tabs, gamma, torch.as_tensor(sb).to(model.device.device), vf, ref,
                                            step_output=out if R == 1 else None)
        rec['cpu_oracle_pairs_per_s'] = extrapolate(timing, B.shape[0], len(vf))['value']
    return rec


def run_config_leg(args) -> dict:
    """
    The other BASELINE configs on one GPU, each point with a parity sample against the oracle:
      configs[0] tiger (S2 A3 O2 R2): the PBVI-RA solve the reference runs on CPU + one backup shape;
      configs[1] 4x4 grid (R = 15 dense and R = 1 no_loop) at B x V in {16, 256, 4096} x {4, 64, 1024};
      configs[4] synthetic random sparse POMDPs; and the sea-robin size (S = 63 555, A = 16, O = 2), the reference's largest workload.
    """
    import torch
    from pomdp_pbvi_exploration_b200 import Model, PBVI_Solver
    from pomdp_pbvi_exploration_b200.recipes import sea_robin_model, synthetic_sparse_model, tiger_model
    rng = np.random.default_rng(0)
    points = []
    # ---- configs[0]
    model = tiger_model()
    seed_all(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vf, hist = PBVI_Solver(0.95, eps=1e-6, expand_function='ra').solve(model, expansions=8, max_belief_growth=10, print_progress=False)
    torch.cuda.synchronize()
    tiger_solve = {'config': 'tiger PBVI-RA solve (expansions=8, max_belief_growth=10)', 'wall_s': time.perf_counter() - t0,
                   'final_alphas': len(vf), 'final_beliefs': int(hist.beliefs_counts[-1]), 'backups': len(hist.backup_times)}
    Bt = _dirichlet_beliefs(rng, 80, 2, 2)
    Vt = np.array([[-100.0, 10.0], [10.0, -100.0], [-1.0, -1.0], [3.0, 5.0], [5.0, 3.0], [-20.0, 8.0], [8.0, -20.0], [0.0, 0.0], [1.0, 2.0]])
    points.append(_config_point('tiger', model, 0.95, Bt, Vt, rng.integers(0, 3, len(Vt)), 50, 80))
    # ---- configs[1]
    for tag in ('grid4x4', 'grid4x4_noloop'):
        m = dict(np.load(os.path.join(ROOT, 'tests', 'golden', f'model_{tag}.npz')))
        S, A, O = m['rto'].shape[0], m['rto'].shape[1], m['rto'].shape[2]
        model = Model(states=S, actions=A, observations=O, transitions=m['transition_table'], rewards=m['reward_table'],
                      observation_table=m['obs_table'], start_probabilities=m['start'])
        for nB in (16, 256, 4096):
            for nV in (4, 64, 1024):
                if tag == 'grid4x4_noloop' and (nB, nV) not in ((256, 64), (4096, 1024)):
                    continue
                B = np.concatenate([np.eye(16)[:min(16, nB)], _dirichlet_beliefs(rng, max(0, nB - 16), 16, 16)])
                V = rng.random((nV, 16)) * 3
                points.append(_config_point(f'{tag} (R={model.reachable_state_count})', model, float(m['gamma']), B, V, rng.integers(0, 4, nV), 20,
                                            256 if nB * nV <= 4096 * 64 else 0))
    # ---- configs[4] + sea-robin size
    for S, A, O, R, parity in ((1000, 4, 2, 1, 256), (10000, 8, 4, 2, 128), (30000, 8, 4, 1, 0), (100000, 16, 8, 4, 0)):
        model = synthetic_sparse_model(S, A, O, R, seed=1)
        B = _dirichlet_beliefs(rng, 1024, S, 2048)
        V = rng.random((256, S))
        points.append(_config_point('synthetic_sparse', model, 0.95, B, V, rng.integers(0, A, 256), 5, parity))
        model.device.close()
        del model
        torch.cuda.empty_cache()
    model = sea_robin_model()
    solver = PBVI_Solver(gamma=GAMMA, eps=1e-8, expand_function='perseus')
    from pomdp_pbvi_exploration_b200 import Belief, ValueFunction
    np.random.seed(4)
    walks = [solver.expand_perseus(model, Belief(model), max_generation=100) for _ in range(10)]
    vf = ValueFunction(model, model.expected_rewards_table.T, model.actions)
    for w in walks[:6]:
        vf = solver.backup(model, w, vf, append=True, belief_dominance_prune=False)
    Bs = torch.cat([w.belief_array for w in walks]).cpu().numpy()
    rec = _config_point('sea_robin (Sea_Robins_Swim_Walk.ipynb)', model, GAMMA, Bs, vf.alpha_vector_array.cpu().numpy(), vf.actions, 5, 48)
    rec['gamma_bytes_the_reference_would_allocate'] = 8.0 * 16 * 2 * rec['V'] * 63555
    points.append(rec)
    bad = [p['config'] for p in points if 'parity_sample' in p and not p['parity_sample']['ok']]
    return {'tiger_solve': tiger_solve, 'points': points, 'parity_failures': bad, 'ssea_expansions': run_ssea_points(rng)}


def run_config_leg_sharded(world: int, rank: int) -> dict:
    """The other BASELINE configs at N > 1: the same belief sets as at N = 1, SHARDED over the ranks (strong scaling).  tiger and the 4x4
    grid are launch- and latency-bound (a few microseconds of arithmetic): more GPUs only add the exchange, and the numbers say so."""
    import torch
    from pomdp_pbvi_exploration_b200 import Belief, Model, PBVI_Solver, ValueFunction
    from pomdp_pbvi_exploration_b200.recipes import sea_robin_model, synthetic_sparse_model, tiger_model
    rng = np.random.default_rng(0)                       # same inputs on every rank
    points = []
    try:
        model = tiger_model()
        Bt = _dirichlet_beliefs(rng, 80, 2, 2)
        Vt = np.array([[-100.0, 10.0], [10.0, -100.0], [-1.0, -1.0], [3.0, 5.0], [5.0, 3.0], [-20.0, 8.0], [8.0, -20.0], [0.0, 0.0], [1.0, 2.0]])
        points.append(_config_point('tiger', model, 0.95, Bt, Vt, rng.integers(0, 3, len(Vt)), 20, 80, world, rank))
        for tag in ('grid4x4', 'grid4x4_noloop'):
            m = dict(np.load(os.path.join(ROOT, 'tests', 'golden', f'model_{tag}.npz')))
            model = Model(states=16, actions=4, observations=2, transitions=m['transition_table'], rewards=m['reward_table'],
                          observation_table=m['obs_table'], start_probabilities=m['start'])
            B = np.concatenate([np.eye(16), _dirichlet_beliefs(rng, 4096 - 16, 16, 16)])
            V = rng.random((1024, 16)) * 3
            points.append(_config_point(f'{tag} (R={model.reachable_state_count})', model, float(m['gamma']), B, V, rng.integers(0, 4, 1024), 10, 64,
                                        world, rank))
        for S, A, O, R, parity in ((10000, 8, 4, 2, 64), (30000, 8, 4, 1, 0)):
            model = synthetic_sparse_model(S, A, O, R, seed=1)
            B = _dirichlet_beliefs(rng, 1024, S, 2048)
            V = rng.random((256, S))
            points.append(_config_point('synthetic_sparse', model, 0.95, B, V, rng.integers(0, A, 256), 5, parity, world, rank))
            model.device.close()
            del model
            torch.cuda.empty_cache()
        model = sea_robin_model()
        solver = PBVI_Solver(gamma=GAMMA, eps=1e-8, expand_function='perseus')
        np.random.seed(4)
        walks = [solver.expand_perseus(model, Belief(model), max_generation=100) for _ in range(10)]
        vf = ValueFunction(model, model.expected_rewards_table.T, model.actions)
        for w in walks[:6]:
            vf = solver.backup(model, w, vf, append=True, belief_dominance_prune=False)
        Bs = torch.cat([w.belief_array for w in walks]).cpu().numpy()
        points.append(_config_point('sea_robin (Sea_Robins_Swim_Walk.ipynb)', model, GAMMA, Bs, vf.alpha_vector_array.cpu().numpy(), vf.actions, 5, 48,
                                    world, rank))
    except Exception as e:                                # (a rank that fails here would leave the others in a collective: report and stop)
        return {'error': f'{type(e).__name__}: {e}', 'points': [p for p in points if p]}
    points = [p for p in points if p]
    bad = [p['config'] for p in points if 'parity_sample' in p and not p['parity_sample']['ok']]
    return {'points': points, 'parity_failures': bad, 'n_gpus': world,
            'note': 'the N = 1 belief sets sharded over the ranks (strong scaling), time = max over ranks'}


def run_ssea_points(rng) -> list:
    """
    SSEA expansions at scale (configs[1] names SSEA on the 4x4 grid; the reference's own expand_ssea crashes on every model that has an
    impossible observation, SURVEY.md section 4): all B*A*O successors from one launch, their distance to the belief set with the tiled
    direct-difference kernel, the `max_generation` farthest kept.  Timed end to end (`PBVI_Solver.expand_ssea`), with the distances of a
    sample of possible successors checked against the reference's formula (oracle.ssea_min_distances).
    """
    import torch
    from oracle import pbvi_oracle as orc
    from pomdp_pbvi_exploration_b200 import BeliefSet, Model, PBVI_Solver
    from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model
    out = []
    m = dict(np.load(os.path.join(ROOT, 'tests', 'golden', 'model_grid4x4.npz')))
    grid = Model(states=16, actions=4, observations=2, transitions=m['transition_table'], rewards=m['reward_table'],
                 observation_table=m['obs_table'], start_probabilities=m['start'])
    olf = olfactory_wrap_model()
    solver = PBVI_Solver(gamma=GAMMA, eps=1e-6, expand_function='ssea')
    np.random.seed(9)
    cases = [('grid4x4 (R=15)', grid, np.concatenate([np.eye(16), _dirichlet_beliefs(rng, 4096 - 16, 16, 16)]), 100),
             ('olfactory_wrap', olf, torch.cat([solver.expand_perseus(olf, __import__('pomdp_pbvi_exploration_b200').Belief(olf), 100).belief_array
                                                for _ in range(10)]).cpu().numpy(), 100)]
    for name, model, B, n_new in cases:
        bs = BeliefSet(model, B)
        dev = model.device
        for _ in range(2):
            new = solver.expand_ssea(model, bs, max_generation=n_new)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        new = solver.expand_ssea(model, bs, max_generation=n_new)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        # parity of the ingredients on a sample: successors of 4 beliefs, distances to the whole set
        pick = np.unique(np.linspace(0, B.shape[0] - 1, 4).astype(np.int64))
        succ, mass = dev.belief_successors(torch.as_tensor(B[pick]).to(dev.device))
        tabs = host_tables(model)
        with np.errstate(all='ignore'):
            want_succ = orc.all_successors(tabs['reach'], tabs['rto'], B[pick])
            ok_succ = bool(np.array_equal(succ.cpu().numpy(), want_succ, equal_nan=True))
            possible = ~np.isnan(want_succ.reshape(-1, B.shape[1])).any(axis=1)
            cand = want_succ.reshape(-1, B.shape[1])[possible]
            want_d = np.array([np.sqrt(np.min(np.einsum('bs,bs->b', B - c, B - c))) for c in cand])
        got_d = dev.min_l2_distance(bs.belief_array, torch.as_tensor(cand).to(dev.device)).cpu().numpy()
        out.append({'config': name, 'S': model.state_count, 'B': int(B.shape[0]), 'candidates': int(B.shape[0] * model.action_count * model.observation_count),
                    'max_generation': n_new, 'new_beliefs': len(new), 'expand_ssea_s': wall,
                    'parity_sample': {'successor_rows_bitwise_equal': ok_succ, 'distances_checked': int(cand.shape[0]),
                                      'max_rel_distance_error': float(np.max(np.abs(got_d - want_d) / np.maximum(want_d, 1e-300))) if cand.shape[0] else 0.0,
                                      'ok': ok_succ and bool(np.allclose(got_d, want_d, rtol=1e-10, atol=1e-13))}})
    return out


_JSON_OUT = None


def emit(line: dict) -> None:
    """The one JSON line goes to the real stdout; everything else printed during the run (NCCL banners, library logs) was
    redirected to stderr by main()."""
    os.write(_JSON_OUT, (json.dumps(line) + '\n').encode())


def main():
    global _JSON_OUT
    a = parse_args()
    sys.stdout.flush()
    _JSON_OUT = os.dup(1)
    os.dup2(2, 1)                      # fd 1 -> stderr for native code too (NCCL prints its version banner on stdout)
    sys.stdout = sys.stderr
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_b200(a)


if __name__ == '__main__':
    main()
