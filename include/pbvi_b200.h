/*
 * pbvi_b200.h -- C ABI of the B200-native PBVI backup engine (libpbvi_b200.so).
 *
 * The reference (PimLb/POMDP_PBVI_Exploration) is pure Python and has no FFI of its own; its "device
 * boundary" is CuPy (`xp = cp.get_array_module(...)`, src/pomdp.py:1482).  The entry points below are
 * what a binding for the hot path would bind: each one replaces the body of one reference method and
 * cites it.  INTEGRATION.md shows the ctypes stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative pbvi_status; the message of the last failure on
 *     the calling thread is returned by pbvi_last_error().  No C++ exception crosses the boundary.
 *   - pointers named d_* are DEVICE pointers on the handle's device, h_* are HOST pointers.  All arrays are
 *     C-contiguous.  Floating data is IEEE binary64, indices int32 unless stated (host model tables use the
 *     reference's int64 `reachable_states`).
 *   - the library BORROWS every pointer for the duration of the call; the only object that outlives a call
 *     is the opaque model handle, which owns the device copy of the model tables and a grow-only scratch arena.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls enqueue work on it and
 *     return without synchronising unless stated otherwise.
 *   - a handle is not re-entrant: one host thread per handle (one process per GPU under torchrun).  Its scratch is reused by
 *     consecutive calls in stream order; a call issued on a different stream than the previous one on the same handle first waits, on
 *     the device, for the work that call enqueued (so switching streams is safe, overlapping two calls of one handle is not possible).
 */
#ifndef PBVI_B200_H
#define PBVI_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define PBVI_API __attribute__((visibility("default")))
#else
#define PBVI_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pbvi_model pbvi_model;

typedef enum pbvi_status {
    PBVI_OK = 0,
    PBVI_ERR_BAD_ARG = -1,
    PBVI_ERR_CUDA = -2,
    PBVI_ERR_OOM = -3,
    PBVI_ERR_UNSUPPORTED = -4,
    PBVI_ERR_NCCL = -5
} pbvi_status;

/* library version (major*100 + minor) and the message of the calling thread's last error */
PBVI_API int pbvi_version(void);
PBVI_API const char* pbvi_last_error(void);

/* ---- model tables --------------------------------------------------------------------------------
 * Replaces Model.gpu_model (src/mdp.py:533-560): uploads the tables the kernels consume, re-laid out
 * action-major.  Host inputs are in the reference's layouts:
 *   h_reach [S][A][R] int64  reachable_states                           (src/mdp.py:296-353)
 *   h_probs [S][A][R] f64    reachable_probabilities (may be NULL: VI sweep then unavailable)
 *   h_rto   [S][A][O][R] f64 reachable_transitional_observation_table   (src/pomdp.py:197-205)
 *   h_rbar  [S][A] f64       expected_rewards_table                     (src/pomdp.py:231-254)
 */
PBVI_API int pbvi_model_create(int S, int A, int O, int R, const int64_t* h_reach, const double* h_probs,
                      const double* h_rto, const double* h_rbar, int device, pbvi_model** out);
PBVI_API int pbvi_model_destroy(pbvi_model* m);
PBVI_API int pbvi_model_dims(const pbvi_model* m, int* S, int* A, int* O, int* R);

/* ---- point-based backup (PBVI_Solver.backup, src/pomdp.py:1447-1524) -------------------------------
 * pbvi_backup_select: steps 1-3 without materialising Gamma.  For every belief b:
 *   v_star[b][a][o] = first index of max_v  belief_b . Gamma[a,o,v]                      (:1489-1495)
 *   value[b][a]     = belief_b . (Rbar[:,a] + sum_o Gamma[a,o,v_star[b][a][o]])          (:1502-1505)
 *   a_star[b]       = first index of max_a value[b][a]                                   (:1505)
 * d_beliefs [nB][S], d_alphas [nV][S]; outputs d_vstar [nB][A][O] int32, d_value [nB][A] (nullable),
 * d_astar [nB] int32.  value[b][a] is summed in the reference's operation order for every action that can win or tie
 * (approximate value within the rounding margin of the best one); actions that cannot win carry their approximate value.
 * With d_value == NULL only a_star is produced, and beliefs with a single possible winner skip the exact sum.
 */
PBVI_API int pbvi_backup_select(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV,
                       double gamma, int32_t* d_vstar, double* d_value, int32_t* d_astar, void* stream);

/* pbvi_backup_assemble: alpha_a rows for n (action, v_star[O]) tuples                    (:1497-1506)
 *   out[i][s] = Rbar[s,a_i] + ((G_0 + G_1) + ...),  G_o = gamma * sum_r RTO[s,a_i,o,r] * alpha[v_i[o]][reach[s,a_i,r]]
 * with the reference's operation order and no FMA contraction (bit-identical rows when R == 1).
 * d_actions [n] int32, d_vsel [n][O] int32, d_out [n][S]; d_hash [n][2] uint64 (nullable) receives the 128-bit key of every
 * row (the value pbvi_row_hash computes), accumulated while the row is being written.
 */
PBVI_API int pbvi_backup_assemble(pbvi_model* m, const double* d_alphas, int nV, double gamma, const int32_t* d_actions,
                         const int32_t* d_vsel, int n, double* d_out, uint64_t* d_hash, void* stream);

/* pbvi_controller_sweep: one evaluation sweep of a finite-state controller (PolicyGraph) with n nodes, node i playing d_actions[i] and
 * moving to node d_succ[i][o] on observation o:
 *   d_out[i][s] = Rbar[s,a_i] + ((G_0 + G_1) + ...),  G_o = gamma * sum_r RTO[s,a_i,o,r] * d_in[succ_i[o]][reach[s,a_i,r]]
 * i.e. bitwise the rows pbvi_backup_assemble(d_in, n, gamma, d_actions, d_succ) gives.  d_in [n][S] must be finite (zero-RTO terms
 * are skipped as for finite alphas); indices are clamped into range.  d_stats3 (nullable) receives, from the same launch,
 * {max(out - in), max(in - out), max |out - in|} over all n*S entries, rows paired by index (NaN wins).
 * Enqueues on `stream`, does not synchronise. */
PBVI_API int pbvi_controller_sweep(pbvi_model* m, const double* d_in, int n, double gamma, const int32_t* d_actions,
                                   const int32_t* d_succ, double* d_out, double* d_stats3, void* stream);

/* pbvi_controller_evaluate: up to max_sweeps sweeps W <- T_pi W of pbvi_controller_sweep from W = d_in in one persistent cooperative
 * launch, stopping after the first sweep whose max |out - in| is below tol or NaN.  d_out [n][S] receives the last iterate (d_in is not
 * written and must not be d_out), d_changes [max_sweeps] (nullable) each sweep's max |out - in|, *h_sweeps the number of sweeps run.
 * k sweeps give bitwise the rows and change values of k pbvi_controller_sweep calls.  Synchronises `stream` once, at the end. */
PBVI_API int pbvi_controller_evaluate(pbvi_model* m, const double* d_in, int n, double gamma, const int32_t* d_actions,
                                      const int32_t* d_succ, double tol, int max_sweeps, double* d_out, double* d_changes,
                                      int* h_sweeps, void* stream);

/* pbvi_backup: select + assemble for every belief (no dedup): d_out_alpha [nB][S], d_out_action [nB];
 * d_out_vstar [nB][A][O] and d_out_value [nB][A] may be NULL. */
PBVI_API int pbvi_backup(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double gamma,
                double* d_out_alpha, int32_t* d_out_action, int32_t* d_out_vstar, double* d_out_value, void* stream);

/* Same with HOST buffers: copies inputs to the device, runs pbvi_backup, copies alpha rows and actions back and
 * synchronises.  This is the end-to-end entry point a CPU-resident caller (the reference's NumPy path) would use.  The beliefs are
 * processed in chunks of 2048 rows through a two-deep pipeline (upload of chunk k + 1 | kernels of chunk k | download of chunk k - 1),
 * so with pinned (page-locked) buffers the call is bound by the PCIe link, not by link + kernels + link; pageable buffers work, unoverlapped. */
PBVI_API int pbvi_backup_host(pbvi_model* m, const double* h_beliefs, int nB, const double* h_alphas, int nV, double gamma,
                     double* h_out_alpha, int32_t* h_out_action, void* stream);

/* The reference's whole `PBVI_Solver.backup` (src/pomdp.py:1447-1524 with belief_dominance_prune = False, append = False) from host
 * buffers in one call -- including what `ValueFunction(model, alpha_vectors, best_actions)` does to the rows (src/mdp.py:668-669: one
 * entry per distinct row, position of the first occurrence, action of the last).  Sparse belief sets of 2048 rows or more travel
 * packed (the library's own host threads pack slabs of rows into pinned staging, pbvi_unpack_rows rebuilds them in HBM behind the
 * copies: the belief buffer may be pageable), others through the chunked upload of pbvi_backup_host; pageable alpha / output buffers
 * pass through pinned staging.  Then the distinct generating tuples (a*, v*[a*, :]) in order of first occurrence, one alpha row per tuple, the
 * byte-dedup of those rows on 128-bit keys (every match confirmed bytewise), and only the surviving rows are copied back:
 * h_out_alpha [*h_n_out][S], h_out_action [*h_n_out].  out_capacity = rows the output buffers hold (nB always suffices); if the result
 * has more, *h_n_out is set and PBVI_ERR_BAD_ARG returned.  PBVI_ERR_UNSUPPORTED: two different rows shared a key (never observed) --
 * call pbvi_backup_host and de-duplicate on the host.  Synchronises. */
PBVI_API int pbvi_backup_host_unique(pbvi_model* m, const double* h_beliefs, int nB, const double* h_alphas, int nV, double gamma,
                            double* h_out_alpha, int out_capacity, int32_t* h_out_action, int* h_n_out, void* stream);

/* pbvi_backup_small: the WHOLE `PBVI_Solver.backup(append=False)` of a small problem (tiger, 4x4 grids: BASELINE configs[0] / [1]) in one
 * call -- one kernel (a block per belief: projections, v*, values, a*, the alpha row and its 128-bit key, all in shared memory), one
 * copy back, the ValueFunction constructor's dict semantics on the host (src/mdp.py:668-669: position of the first occurrence, action
 * of the last; key matches confirmed with memcmp) and a gather of the surviving rows.  d_out_rows has room for nB rows; the first
 * *h_n_out are written (stream-ordered), h_out_actions [nB] / h_out_keys [nB][2] (nullable) receive their actions and row keys.
 * Synchronises `stream` once.  pbvi_backup_small_eligible tells whether the sizes qualify (everything of one belief in shared memory,
 * at most ~6e7 multiply-adds); otherwise PBVI_ERR_UNSUPPORTED: use pbvi_backup_select / pbvi_backup_assemble. */
PBVI_API int pbvi_backup_small_eligible(const pbvi_model* m, int nB, int nV);
PBVI_API int pbvi_backup_small(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double gamma,
                               double* d_out_rows, int32_t* h_out_actions, uint64_t* h_out_keys, int* h_n_out, void* stream);

/* ---- maxima over a value function (src/pomdp.py:2165-2167 compute_change, :1639 SSGA, :1735 GER, :1393) ----
 * d_max[b] = max_v belief_b . alpha_v, d_arg[b] = its first index.  Either output may be NULL. */
PBVI_API int pbvi_max_values(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV,
                    double* d_max, int32_t* d_arg, void* stream);

/* ---- belief update (Belief.update, src/pomdp.py:382-421; batched twin :1415-1419) ----------------
 * out[i][s'] = sum_{(s,r): reach[s,a_i,r]=s'} RTO[s,a_i,o_i,r] * belief_i[s], accumulated in ascending (s,r) order like
 * bincount, then divided by its NumPy-pairwise sum when `normalise` != 0 (0/0 = NaN for impossible observations, as
 * in the reference).  d_norm[i] (nullable) receives the un-normalised mass P(o_i | b_i, a_i).
 */
PBVI_API int pbvi_belief_update(pbvi_model* m, const double* d_beliefs, const int32_t* d_actions, const int32_t* d_observations,
                       int n, int normalise, double* d_out, double* d_norm, void* stream);

/* A chain of n updates from d_b0 (the FSVI / FSVI_EG trajectory, src/pomdp.py:1905-1930): d_out[i] = update(prev_i, a_i, o_i) with
 * prev_0 = d_b0 and prev_{i+1} = d_out[i], or d_b0 again when h_reset[i] != 0 (end state reached: restart from b0).  The (a,o)
 * sequence comes from the host RNG walk and is passed in HOST arrays; 2n launches are enqueued, nothing is read back. */
PBVI_API int pbvi_belief_trajectory(pbvi_model* m, const double* d_b0, const int32_t* h_actions, const int32_t* h_observations,
                                    const uint8_t* h_reset, int n, double* d_out, void* stream);

/* The Perseus random walk in belief space (PBVI_Solver.expand_perseus, src/pomdp.py:2040-2054): for i < n, a_i = h_actions[i] (drawn on the
 * host, `np.random.choice(model.actions)`), o_i ~ P(o | b_i, a_i) drawn ON THE DEVICE from the host's uniform h_uniforms[i] exactly as
 * `np.random.choice(observations, p=obs_prob)` does (cdf = cumsum(p) / cumsum(p)[-1]; searchsorted(cdf, u, 'right') -- that call
 * consumes one `random_sample()`, so pre-drawing (a_i, u_i) in this order leaves the reference's RNG stream unchanged), and
 * d_out[i] = b_{i+1} = update(b_i, a_i, o_i), b_0 = d_b0.  d_observations [n] (nullable) receives the o_i.  4n launches are
 * enqueued and nothing is read back: the host-driven form pays two synchronisations per step. */
PBVI_API int pbvi_perseus_walk(pbvi_model* m, const double* d_b0, const int32_t* h_actions, const double* h_uniforms, int n,
                               double* d_out, int32_t* d_observations, void* stream);

/* Every successor of every belief (Belief.generate_successors, src/pomdp.py:424-438; the B*A*O loop of SSEA :1679 and
 * GER :1732): d_out [n][A][O][S], d_norm [n][A][O] (nullable).  Rows of impossible observations are NaN when normalised. */
PBVI_API int pbvi_belief_successors(pbvi_model* m, const double* d_beliefs, int n, int normalise, double* d_out, double* d_norm, void* stream);

/* P(o | b, a) for every (a,o): d_out [n][A][O]  (einsum 'sor,s->o', src/pomdp.py:1814, 2046; 'bs,saor->bao' :1751) */
PBVI_API int pbvi_observation_probabilities(pbvi_model* m, const double* d_beliefs, int n, double* d_out, void* stream);

/* ---- raw-byte set semantics (src/mdp.py:668-669, 773-774; src/pomdp.py:581,600) --------------------
 * pbvi_row_hash: 128-bit hash of the raw bytes of each row, d_hash [n][2] uint64.
 * pbvi_rows_equal: flags[i] = 1 iff rows_a[ia[i]] and rows_b[ib[i]] are bytewise identical (used to confirm hash matches,
 * so the dedup is exact, not probabilistic). */
PBVI_API int pbvi_row_hash(pbvi_model* m, const double* d_rows, int n, int row_len, uint64_t* d_hash, void* stream);
PBVI_API int pbvi_rows_equal(pbvi_model* m, const double* d_rows_a, const int32_t* d_ia, const double* d_rows_b, const int32_t* d_ib,
                    int n, int row_len, int32_t* d_flags, void* stream);

/* pbvi_group_keys: the insertion order of the reference's `{row.tobytes(): alpha_vector}` dicts (ValueFunction ctor
 * src/mdp.py:668-669; BeliefSet src/pomdp.py:581,600) for n fixed-width keys, computed on the device: the (a*, v*[a*,:]) tuples
 * of a backup and the 128-bit keys of its alpha rows are grouped without leaving HBM.  d_keys [n][words] uint32.  Groups are
 * numbered by first occurrence; d_first[g] = index of the group's first record (ascending in g), d_last[g] = index of its
 * record with the largest (d_rank[i], i) -- the last occurrence when d_rank is NULL ("first position, last action") --,
 * d_inverse[i] (nullable) = group of record i.  d_first / d_last have room for n entries; *h_count receives the number of
 * groups.  Synchronises `stream`. */
PBVI_API int pbvi_group_keys(pbvi_model* m, const uint32_t* d_keys, int n, int words, const int32_t* d_rank, int32_t* d_first,
                    int32_t* d_last, int32_t* d_inverse, int* h_count, void* stream);

/* pbvi_group_record_blocks: the merge step of the sharded backup's tuple exchange (all-gather of each rank's new alpha vectors,
 * in generating-tuple form).  d_blocks is the gathered buffer: `world` blocks of block_rows rows of (words + 2) int32; row 0 of a
 * block is its header (word 0 = number of records u_r of rank r), rows 1..u_r are records (key[words], first position, last
 * position).  Records are grouped by key in buffer order (rank-major = belief order), like one dict over the whole belief set:
 * d_first[g] = row of the group's first record, d_last[g] = row of its record with the largest last position (rows index the
 * whole buffer; outputs have room for world*block_rows entries).  *h_count = number of groups, *h_max_records = max_r u_r
 * (a value above block_rows - 1 means a rank overflowed its block: repeat the exchange with larger blocks).  Synchronises. */
PBVI_API int pbvi_group_record_blocks(pbvi_model* m, const int32_t* d_blocks, int world, int block_rows, int words, int32_t* d_first,
                             int32_t* d_last, int* h_count, int* h_max_records, void* stream);

/* pbvi_confirm_groups: *h_all_equal = 1 iff every row equals, bytewise, the first row of its group (d_first, d_inverse from
 * pbvi_group_keys over the rows' 128-bit keys): makes the key-based dedup exact.  Synchronises `stream`. */
PBVI_API int pbvi_confirm_groups(pbvi_model* m, const double* d_rows, int n, int row_len, const int32_t* d_first,
                        const int32_t* d_inverse, int* h_all_equal, void* stream);

/* ---- host -> device transport of sparse rows (the reference's GPU path copies the dense belief array: Model.gpu_model /
 * `cp.array(belief_array)`, src/pomdp.py:1482) ---------------------------------------------------------------------------
 * pbvi_pack_rows_host (pure host code, thread-safe, no handle): packs n rows of row_len doubles into a bitmap over 4-double
 * chunks (h_bitmap [n][W] uint32, W = ceil(ceil(row_len/4)/32)), the chunks that contain a non-zero BIT (so -0.0 survives)
 * back to back in h_packed (room for n*ceil(row_len/4)*4 doubles) and the first chunk of every row in h_row_start [n+1];
 * *h_chunks = number of chunks written (h_packed needs one chunk of slack beyond that).  Rows are packed in slabs (one call per
 * slab, slabs in parallel on host threads).  pbvi_unpack_rows rebuilds n dense rows [n][row_len] in device memory from device
 * copies of the arrays of consecutive slabs of slab_rows rows each, byte for byte: row i belongs to slab i / slab_rows, whose
 * chunks start at slab * region_chunks in d_packed and whose row offsets are d_row_start[slab * (slab_rows + 1) + i % slab_rows]. */
PBVI_API int pbvi_pack_rows_host(const double* h_rows, int n, int row_len, uint32_t* h_bitmap, int32_t* h_row_start, double* h_packed,
                        int64_t* h_chunks);
/* One packer thread's share of a row set: slabs first_slab, first_slab + slab_step, ... (slab i = rows [i*slab_rows, ...)); slab i's
 * chunks go to h_packed + i*region_doubles, its offsets to h_row_start + i*(slab_rows+1) and, last, its chunk count to h_totals[i]
 * (release store; initialise to -1 and poll: -2 = failed). */
PBVI_API int pbvi_pack_slabs_host(const double* h_rows, int n, int row_len, int slab_rows, int first_slab, int slab_step, uint32_t* h_bitmap,
                         int32_t* h_row_start, double* h_packed, int64_t region_doubles, int64_t* h_totals);
PBVI_API int pbvi_unpack_rows(pbvi_model* m, const uint32_t* d_bitmap, const int32_t* d_row_start, const double* d_packed, int n,
                     int row_len, int slab_rows, int64_t region_chunks, double* d_out, void* stream);

/* ---- MDP value iteration sweep (src/mdp.py:1507) ---------------------------------------------------
 * d_alpha_out[a][s] = Rbar[s,a] + gamma * sum_r P[s,a,r] * d_vopt[reach[s,a,r]];  d_vopt_out[s] = max_a (nullable) */
PBVI_API int pbvi_vi_sweep(pbvi_model* m, const double* d_vopt, double gamma, double* d_alpha_out, double* d_vopt_out, void* stream);

/* ---- Fast Informed Bound sweep (Hauskrecht 2000; FIB_Solver) ------------------------------------------------------------------------
 * d_out[a][s] = Rbar[s,a] + gamma * sum_o max_{a' < k} sum_r RTO[s,a,o,r] * d_in[a'][reach[s,a,r]]   for k input rows d_in [k][S],
 * A output rows.  Fixed order (r ascending, then o ascending, no fma contraction): R = 1 models reproduce a NumPy restatement bit for bit.
 * d_stats2 (nullable; needs k == A, rows paired by index) receives {max(out - in), max |out - in|} from the same launch (NaN wins).
 * Enqueues on `stream`, does not synchronise. */
PBVI_API int pbvi_fib_sweep(pbvi_model* m, const double* d_in, int k, double gamma, double* d_out, double* d_stats2, void* stream);

/* ---- pointwise-domination prune (ValueFunction.prune level 2, src/mdp.py:857-866) -------------------
 * d_keep[i] = 1 iff alpha_i is >= everywhere by no vector other than itself. */
PBVI_API int pbvi_prune_dominated(pbvi_model* m, const double* d_alphas, int nV, int32_t* d_keep, void* stream);

/* pbvi_first_dominating_row: domination of one row set by another (the improvement step of policy iteration on a controller).
 * d_first[i] = the smallest j with d_new[j][s] >= d_old[i][s] at every state s (a NaN on either side fails), or -1; rows have length S.
 * Equal rows dominate.  Enqueues on `stream`, does not synchronise. */
PBVI_API int pbvi_first_dominating_row(pbvi_model* m, const double* d_new, int n_new, const double* d_old, int n_old, int32_t* d_first,
                                       void* stream);

/* ---- LP-domination prune (ValueFunction.prune level 3; the reference's intended Lark / White filter, src/mdp.py:834-906, whose
 * branch fails on the undefined `pruned_alpha_set` at :872) ----------------------------------------------------------------------
 * d_keep[i] = 0 iff a convex combination of the other rows exceeds alpha_i by more than tol = 1e-9*max(1, max|alpha|) at every
 * state (verified in FP64); d_bound[i] (nullable) = the verified bound behind the decision (witness margin lower bound m* for kept
 * rows, certificate upper bound u for pruned ones); h_counts[4] (nullable) = {kept at a corner, kept by an LP witness, pruned,
 * kept undecided}.  Rows must be pairwise distinct.  A row with a non-finite entry is kept (counted with the corners, bound NaN) and
 * never used as a competitor.  Synchronises `stream`. */
PBVI_API int pbvi_prune_lp(pbvi_model* m, const double* d_alphas, int nV, int32_t* d_keep, double* d_bound, int32_t* h_counts, void* stream);
/* instrumentation of the last pbvi_prune_lp call: h_out4 = {largest competitor set |J| reached, restricted LPs solved, simplex pivots,
 * rows sent to the LP stage} */
PBVI_API int pbvi_prune_lp_stats(const pbvi_model* m, int64_t* h_out4);

/* ---- HSVI sawtooth upper bound (BeliefValueMapping.evaluate, src/pomdp.py:887-895) -----------------
 * d_out[q] = min(v0_q, min_i v0_q + (ub_value_i - ub_belief_i . corner) * min_{s: ub_belief_i[s] > 0} query_q[s]/ub_belief_i[s]) */
PBVI_API int pbvi_sawtooth(pbvi_model* m, const double* d_corner, const double* d_ub_beliefs, const double* d_ub_values, int n_ub,
                  const double* d_queries, int n_q, double* d_out, void* stream);

/* Stored beliefs as SUPPORT LISTS (built once when a belief enters the upper-bound arrays): for row i, d_idx / d_val [i*S, i*S + d_count[i])
 * hold the states and values of its positive entries, d_dot[i] = row_i . corner.  pbvi_sawtooth_lists is pbvi_sawtooth over such lists
 * (same values: the minimum runs over the support either way); a level then touches nnz instead of S entries per stored belief. */
PBVI_API int pbvi_support_lists(pbvi_model* m, const double* d_rows, int n, const double* d_corner, int32_t* d_idx, double* d_val,
                                int32_t* d_count, double* d_dot, void* stream);
PBVI_API int pbvi_sawtooth_lists(pbvi_model* m, const double* d_corner, const int32_t* d_idx, const double* d_val, const int32_t* d_count,
                                 const double* d_dot, const double* d_ub_values, int n_ub, const double* d_queries, int n_q, double* d_out,
                                 void* stream);

/* ---- one level of HSVI's exploration (PBVI_Solver.expand_hsvi, src/pomdp.py:1803-1855) in one call, one synchronisation ---------------
 * For the belief d_b: all A*O successors (d_succ [A][O][S], NaN rows for impossible observations) and masses P(o|b,a) (d_mass [A][O]; both
 * nullable: scratch is used when the caller does not want them);
 * their upper bounds -- the stored value when the successor's 128-bit key is among d_stored_keys [n_stored][2] (:884-885), else the
 * sawtooth over the n_ub stored beliefs of the support lists (the arrays as of the last BeliefValueMapping.update, :866-871) --;
 * Q(a) = b.Rbar[:,a] + gamma * sum_o P(o|b,a) * upper(a,o) and a = its first argmax (:1807-1821); max_v alpha_v . successor as the lower
 * bound; o = first argmax of P(o|b,a) * (upper - lower) (:1826-1842); observations of probability zero are skipped.  When may_continue
 * != 0, upper - lower >= conv_term and key(b) is not stored yet, (key(b), Q(a)) is appended at index n_stored of the stored arrays
 * (:1849).  d_next [S] (nullable) receives the chosen successor update(b, a, o) -- b itself when no observation is possible.  h_out8 receives {best_a, best_o, Q(a), upper - lower} as doubles followed by {added, key0(b), key1(b), #possible (a,o)} as
 * int64.  Synchronises `stream`. */
PBVI_API int pbvi_hsvi_level(pbvi_model* m, const double* d_b, const double* d_alphas, int nV, double gamma, const double* d_corner,
                             const int32_t* d_idx, const double* d_val, const int32_t* d_count, const double* d_dot,
                             const double* d_ub_values, int n_ub, uint64_t* d_stored_keys, double* d_stored_vals, int n_stored,
                             int stored_capacity, double conv_term, int may_continue, double* d_next, double* d_succ, double* d_mass,
                             double* h_out8, void* stream);

/* ---- point-based upper-bound backup of n beliefs (UpperBound.improve) ------------------------------------------------------------------
 * The bound is min(F, sawtooth): F(b) = max_{a < k} d_fib[a] . b over k upper-bound rows d_fib [k][S] (FIB rows), and the sawtooth over the
 * n_ub stored beliefs of the support lists (as for pbvi_sawtooth_lists; d_corner = max_a d_fib[a][s]).  For every belief b_i of d_b [n][S]:
 *   d_u[i]      = max_a [ b_i.Rbar[:,a] + gamma * sum_{o: P(o|b_i,a) > 0} P(o|b_i,a) * min(F, sawtooth)(b_i^{ao}) ]   (o ascending)
 *   d_cur[i]    = min(F, sawtooth)(b_i)           (nullable)
 *   d_best_a[i] = the first maximising action     (nullable)
 * Scratch (n*A*O*S successors, n*A*O*(n_ub+1) sawtooth terms) comes from the handle's arena: the caller sizes n.  Enqueues on `stream`,
 * does not synchronise. */
PBVI_API int pbvi_upper_backup(pbvi_model* m, const double* d_b, int n, const double* d_fib, int k, double gamma, const double* d_corner,
                               const int32_t* d_idx, const double* d_val, const int32_t* d_count, const double* d_dot,
                               const double* d_ub_values, int n_ub, double* d_u, double* d_cur, int32_t* d_best_a, void* stream);

/* ---- one level of K gap-driven trials (GapSolver) -----------------------------------------------------------------------------------
 * For every trial belief b_k of d_b [K][S], with the upper bound of pbvi_upper_backup (d_fib [k][S], corner values, support lists) and
 * the lower bound max_n d_lower[n] . b over N rows d_lower [N][S]:
 *   Q*_k, a*_k  = pbvi_upper_backup's d_u / d_best_a on the same inputs (bitwise: the same launches)
 *   U_o = min(F, sawtooth)(b_k^{a* o}), L_o = max_n d_lower[n] . b_k^{a* o} and e_o = P_o * ((U_o - L_o) - theta) for every o with
 *   P_o = P(o|b_k,a*) > 0 (one rounding per operation; L through the pbvi_max_values path on the O successors of a* only);
 *   o*_k        = without d_uniform or with d_uniform[k] < 0: the first argmax of e over {o : e_o > 0};
 *                 otherwise drawn from that set with weights e_o by NumPy's rule with the uniform d_uniform[k] (as pbvi_perseus_walk
 *                 draws an observation: cdf = cumsum(w), cdf /= cdf[-1], searchsorted(cdf, u, 'right'));
 *                 -1 when no e_o is positive (the trial ends).
 * d_out4 [K][4] receives {a*, o*, Q*, e_{o*}} as doubles (with o* = -1: the largest e_o of a possible o, -inf when there is none);
 * d_next [K][S] the next belief b_k^{a* o*}, bitwise pbvi_belief_update(b_k, a*, o*, normalise = 1) (b_k itself when o* = -1);
 * d_U / d_L [K][O] (nullable, together) U_o and L_o, NaN for impossible observations.  d_uniform [K] is a device array (nullable).
 * Scratch from the handle's arena: K*A*O*S successors, K*A*O*(n_ub + 1) sawtooth terms and K*O*S rows for L: the caller sizes K.
 * Enqueues on `stream`, does not synchronise. */
PBVI_API int pbvi_gap_trial_step(pbvi_model* m, const double* d_b, int K, const double* d_lower, int N, const double* d_fib, int k,
                                 double gamma, const double* d_corner, const int32_t* d_idx, const double* d_val, const int32_t* d_count,
                                 const double* d_dot, const double* d_ub_values, int n_ub, double theta, const double* d_uniform,
                                 double* d_out4, double* d_next, double* d_U, double* d_L, void* stream);

/* ---- SSEA novelty score (src/pomdp.py:1682-1686)--------------------------------------------------
 * d_out[j] = min_i || d_beliefs[i] - d_candidates[j] ||_2 */
PBVI_API int pbvi_min_l2_distance(pbvi_model* m, const double* d_beliefs, int nB, const double* d_candidates, int nC, double* d_out,
                         void* stream);

/* ---- GER error terms (src/pomdp.py:1738-1748) ----------------------------------------------------
 * d_eps[i][a][o] = sum_s (alpha'[s] - d_alpha_b[i][s]) * (d_succ[i][a][o][s] - d_beliefs[i][s]),  alpha'[s] = r_max where the
 * successor gained mass and r_min elsewhere; 0 for the NaN successor of an impossible observation. */
PBVI_API int pbvi_ger_scores(pbvi_model* m, const double* d_beliefs, const double* d_alpha_b, const double* d_succ, int n,
                             double r_min, double r_max, double* d_eps, void* stream);

/* ---- collectives of the belief-sharded path (north_star item 4; reference loop src/pomdp.py:2306-2389) -----------------------------------
 * One process (or thread) per GPU, each with its own pbvi_model and one pbvi_comm.  NCCL is bound with dlopen("libnccl.so.2") on first
 * use (PBVI_NCCL_LIB overrides the name); without it these calls return PBVI_ERR_UNSUPPORTED and everything else keeps working.
 *   pbvi_comm_unique_id   rank 0 creates the 128-byte id and hands it to the other ranks by any host-side means
 *   pbvi_comm_init        collective: every rank calls it with the same id
 *   pbvi_allgather_tuples the exchange step after a local select: every rank contributes one block of block_rows rows of row_words
 *                         int32 -- [header row (record count); records (a*, v*[a*, 0..O-1], first position, last position); padding] --
 *                         and receives the `nranks` blocks in rank order, ready for pbvi_group_record_blocks; every rank then assembles
 *                         the merged tuples itself (pbvi_backup_assemble), so alpha vectors cross NVLink as 4*(3+O) bytes, not 8*S
 *   pbvi_allgather_rows   the literal form: n_rows rows of row_len doubles per rank (pad to a common n_rows)
 *   pbvi_allreduce_max    in-place max over ranks of n doubles (the scalar of compute_change, src/pomdp.py:2165-2169)
 *   pbvi_broadcast_rows   in-place broadcast of `count` doubles from `root` (rank-0 expansion: the new belief rows)
 * All of them enqueue on `stream` and return without synchronising. */
typedef struct pbvi_comm pbvi_comm;
PBVI_API int pbvi_comm_unique_id(unsigned char* id128);
PBVI_API int pbvi_comm_init(pbvi_model* m, const unsigned char* id128, int rank, int nranks, pbvi_comm** out);
PBVI_API int pbvi_comm_destroy(pbvi_comm* c);
PBVI_API int pbvi_comm_rank(const pbvi_comm* c, int* rank, int* nranks);
PBVI_API int pbvi_allgather_tuples(pbvi_comm* c, const int32_t* d_block, int block_rows, int row_words, int32_t* d_gathered, void* stream);
PBVI_API int pbvi_allgather_rows(pbvi_comm* c, const double* d_rows, int n_rows, int row_len, double* d_gathered, void* stream);
PBVI_API int pbvi_allreduce_max(pbvi_comm* c, double* d_values, int n, void* stream);
PBVI_API int pbvi_broadcast_rows(pbvi_comm* c, double* d_rows, size_t count, int root, void* stream);

/* ---- instrumentation: flops actually issued by the last pbvi_backup_select / pbvi_max_values score launch, its grid size
 * and kernel launch count of the last call (for bench.py's roofline / gpu_launches accounting) */
PBVI_API int pbvi_last_stats(const pbvi_model* m, double* executed_flops, double* dense_flops, int* launches);

/* engine options (A/B runs, tests): "chain_kernel" = 2 (default) runs pbvi_belief_trajectory / pbvi_perseus_walk as ONE persistent launch
 * on a thread-block cluster of 8 blocks when a belief fits in shared memory, 1 = the same in one block, 0 = one launch per step-kernel.
 * All three give the same bytes (olfactory model: 20 / 37 / 62 us per step of a Perseus walk). */
PBVI_API int pbvi_set_option(pbvi_model* m, const char* name, int value);

/* kernels launched by the last API call on this handle (host-side counter, no synchronisation) */
PBVI_API int pbvi_last_launches(const pbvi_model* m);

/* pbvi_set_profiling(m, 1): bracket the score kernel launch(es) of every following pbvi_backup* / pbvi_max_values call with CUDA
 * events on the caller's stream; pbvi_last_score_ms waits for the closing event and returns the device time between them
 * (the GEMM-with-argmax launch, plus the Gamma projection for reachable_state_count > 1 models). */
PBVI_API int pbvi_set_profiling(pbvi_model* m, int enable);
PBVI_API int pbvi_last_score_ms(pbvi_model* m, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* PBVI_B200_H */
