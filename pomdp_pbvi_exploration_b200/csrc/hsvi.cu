// One level of HSVI's exploration on the device (reference PBVI_Solver.expand_hsvi, src/pomdp.py:1803-1855, and the sawtooth upper bound
// BeliefValueMapping.evaluate, :873-895).  The reference -- and this package's first version -- walks a level with a host loop over
// (a, o): successor, upper bound, Q-value, then the lower bound of the chosen action's successors: six host round trips per level, 3 ms
// each on the olfactory model.  pbvi_hsvi_level enqueues the whole level and returns with ONE synchronisation:
//     all A*O successors of b with their masses P(o|b,a)                 (belief.cu, one projection launch + one normaliser launch)
//     their 128-bit keys and the key of b                                (stored beliefs return their stored value, :884-885)
//     the sawtooth upper bound of every successor over the stored beliefs (support lists built once per expansion, below)
//     max_v alpha_v . successor for every successor                      (the score kernel, plain path)
//     Q(a) = b.Rbar[:,a] + gamma * sum_o P(o|b,a) * upper(a,o); a = first argmax; o = first argmax of P(o|b,a) * (upper - lower)
//     and, when the recursion goes on, the append of (key(b), Q(a)) to the stored keys / values
// Stored beliefs are kept as SUPPORT LISTS (pbvi_support_lists: states and values of the non-zero entries, and b_i . corner), built once
// when a belief enters the upper-bound arrays instead of being re-compacted by every level: a level then touches nnz, not S, per stored belief.
#include <algorithm>

#include "pbvi_common.cuh"

namespace pbvi {

// ---- support lists (ELL layout: row i owns idx / val [i*S, i*S + count[i])) + dot[i] = row_i . corner -------------------------------
//      The dot product is summed exactly like sawtooth_terms_kernel did (per-thread strided fma, shuffle tree, 8 partials in order),
//      so the upper bounds do not change by a bit.
__global__ void __launch_bounds__(256) support_lists_kernel(const double* __restrict__ rows, const double* __restrict__ corner, int S,
                                                            int32_t* __restrict__ idx, double* __restrict__ val, int32_t* __restrict__ count,
                                                            double* __restrict__ dot) {
    __shared__ double sh[8];
    __shared__ int scount;
    const int i = blockIdx.x;
    const double* r = rows + (size_t)i * S;
    if (threadIdx.x == 0) scount = 0;
    __syncthreads();
    double d = 0.0;
    for (int s0 = 0; s0 < S; s0 += 256) {
        const int s = s0 + threadIdx.x;
        const double b = s < S ? r[s] : 0.0;
        if (s < S) d = fma(b, corner[s], d);
        const bool nz = b > 0.0;
        const unsigned bal = __ballot_sync(0xffffffffu, nz);
        int base = 0;
        if ((threadIdx.x & 31) == 0 && bal) base = atomicAdd(&scount, __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (nz) {
            const int at = base + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u));
            idx[(size_t)i * S + at] = s;
            val[(size_t)i * S + at] = b;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) d += __shfl_down_sync(0xffffffffu, d, off);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = d;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; w++) t += sh[w];
        dot[i] = t;
        count[i] = scount;
    }
}

// terms[q][i] = v0[q] + (ubV[i] - dot[i]) * min_j queries[q][idx_ij] / val_ij ; block per stored belief, Q_TILE queries at a time held
// in registers (the minimum is order-free; the division is the exact one of the reference)
constexpr int SAW_QT = 8;

__global__ void __launch_bounds__(256) sawtooth_lists_kernel(const int32_t* __restrict__ idx, const double* __restrict__ val,
                                                             const int32_t* __restrict__ count, const double* __restrict__ dot,
                                                             const double* __restrict__ ubV, int nUb, const double* __restrict__ queries, int nQ,
                                                             int S, const double* __restrict__ v0, const double* __restrict__ qMass,
                                                             double* __restrict__ terms) {
    __shared__ double sh[8][SAW_QT];
    __shared__ unsigned s_hit;
    const int i = blockIdx.x;
    const int32_t* li = idx + (size_t)i * S;
    const double* lv = val + (size_t)i * S;
    const int cnt = count[i];
    const double scale = ubV[i] - dot[i];
    for (int q0 = 0; q0 < nQ; q0 += SAW_QT) {
        double r[SAW_QT];
        unsigned live = 0u;                       // queries of the tile that exist and (qMass given) have positive mass: NaN rows are skipped
#pragma unroll
        for (int k = 0; k < SAW_QT; k++) {
            r[k] = INFINITY;
            if (q0 + k < nQ && (!qMass || qMass[q0 + k] > 0.0)) live |= 1u << k;
        }
        // Queries and stored beliefs are non-negative, so a ratio of 0 is the floor of the minimum: once every query of the tile has
        // hit a state of the support where it is zero -- the rule: two beliefs of a 22 021-state model rarely nest -- the rest of the list
        // cannot change the result.  (A NaN query, the 0/0 successor of an impossible observation, never reaches 0 and walks the whole
        // list unless the caller passes the masses, which mark it as not live.)  s_hit collects, per query of the tile, "some thread holds a 0".
        if (threadIdx.x == 0) s_hit = 0u;
        __syncthreads();
        const unsigned full = (1u << SAW_QT) - 1u;
        for (int j0 = 0; j0 < cnt; j0 += 256 * 4) {
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int j = j0 + u * 256 + threadIdx.x;
                if (j < cnt) {
                    const int s = li[j];
                    const double b = lv[j];
#pragma unroll
                    for (int k = 0; k < SAW_QT; k++)
                        if ((live >> k) & 1u) r[k] = fmin(r[k], queries[(size_t)(q0 + k) * S + s] / b);
                }
            }
            unsigned hit = ~live & full;
#pragma unroll
            for (int k = 0; k < SAW_QT; k++) hit |= (r[k] == 0.0) ? (1u << k) : 0u;
            hit = __reduce_or_sync(0xffffffffu, hit);
            if ((threadIdx.x & 31) == 0 && hit) atomicOr(&s_hit, hit);
            __syncthreads();
            const bool done = s_hit == full;
            __syncthreads();
            if (done) break;
        }
#pragma unroll
        for (int k = 0; k < SAW_QT; k++) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) r[k] = fmin(r[k], __shfl_down_sync(0xffffffffu, r[k], off));
        }
        __syncthreads();
        if ((threadIdx.x & 31) == 0) {
#pragma unroll
            for (int k = 0; k < SAW_QT; k++) sh[threadIdx.x >> 5][k] = r[k];
        }
        __syncthreads();
        if (threadIdx.x < SAW_QT && q0 + threadIdx.x < nQ) {
            double m = INFINITY;
            for (int w = 0; w < 8; w++) m = fmin(m, sh[w][threadIdx.x]);
            const int q = q0 + threadIdx.x;
            terms[(size_t)q * (nUb + 1) + i] = v0[q] + scale * m;
        }
    }
}

// v0[q] = queries[q] . corner (same reduction shape as sawtooth_v0_kernel); also terms[q][nUb] = v0[q]
__global__ void __launch_bounds__(256) sawtooth_v0_terms_kernel(const double* __restrict__ corner, const double* __restrict__ queries, int S, int nUb,
                                                                double* __restrict__ v0, double* __restrict__ terms) {
    __shared__ double sh[8];
    const double* q = queries + (size_t)blockIdx.x * S;
    double a = 0.0;
    for (int s = threadIdx.x; s < S; s += 256) a = fma(q[s], corner[s], a);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) a += __shfl_down_sync(0xffffffffu, a, off);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; w++) t += sh[w];
        v0[blockIdx.x] = t;
        terms[(size_t)blockIdx.x * (nUb + 1) + nUb] = t;
    }
}

__global__ void __launch_bounds__(128) row_min_lists_kernel(const double* __restrict__ terms, int n, int width, double* __restrict__ out) {
    const int qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= n) return;
    double best = INFINITY;
    for (int i = 0; i < width; i++) best = fmin(best, terms[(size_t)qi * width + i]);
    out[qi] = best;
}

// rb[a] = b . Rbar[:,a] over the non-zero rewards (warp per action)
__global__ void __launch_bounds__(256) reward_dot_kernel(const double* __restrict__ b, const int32_t* __restrict__ nzPtr, const int32_t* __restrict__ nzIdx,
                                                         const double* __restrict__ nzVal, int A, double* __restrict__ rb) {
    const int a = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (a >= A) return;
    double part = 0.0;
    for (int j = nzPtr[a] + lane; j < nzPtr[a + 1]; j += 32) part = fma(b[nzIdx[j]], nzVal[j], part);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) part += __shfl_down_sync(0xffffffffu, part, off);
    if (lane == 0) rb[a] = part;
}

// scores[j][v] = rows[j] . alphas[v] for a FEW rows (the A*O successors of one belief) against all alphas, straight from the row-major
// alphas: block = 8 alphas x 8 rows, thread t owns the states t, t + 256, ... (coalesced loads of both operands), 64 accumulators, fixed
// reduction tree.  The score kernel would run this shape on two SMs (one z, one belief tile: a tile walks its ~1400 pipeline stages
// alone, 0.7 ms); here V / 8 * ceil(n / 8) blocks share the work.  few_rows_max_kernel then takes max_v per row (np.max semantics: NaN wins).
constexpr int FR_A = 8, FR_B = 8;

__global__ void __launch_bounds__(256) few_rows_scores_kernel(const double* __restrict__ rows, int n, const double* __restrict__ alphas, int nV, int S,
                                                              double* __restrict__ scores) {
    __shared__ double sh[8][FR_A * FR_B];
    const int v0 = blockIdx.x * FR_A, j0 = blockIdx.y * FR_B;
    double acc[FR_A][FR_B];
#pragma unroll
    for (int a = 0; a < FR_A; a++)
#pragma unroll
        for (int b = 0; b < FR_B; b++) acc[a][b] = 0.0;
    for (int s = threadIdx.x; s < S; s += 256) {
        double av[FR_A], bv[FR_B];
#pragma unroll
        for (int a = 0; a < FR_A; a++) av[a] = (v0 + a < nV) ? alphas[(size_t)(v0 + a) * S + s] : 0.0;
#pragma unroll
        for (int b = 0; b < FR_B; b++) bv[b] = (j0 + b < n) ? rows[(size_t)(j0 + b) * S + s] : 0.0;
#pragma unroll
        for (int a = 0; a < FR_A; a++)
#pragma unroll
            for (int b = 0; b < FR_B; b++) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
    }
#pragma unroll
    for (int a = 0; a < FR_A; a++)
#pragma unroll
        for (int b = 0; b < FR_B; b++) {
            double x = acc[a][b];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) x += __shfl_down_sync(0xffffffffu, x, off);
            if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5][a * FR_B + b] = x;
        }
    __syncthreads();
    if (threadIdx.x < FR_A * FR_B) {
        double t = 0.0;
        for (int w = 0; w < 8; w++) t += sh[w][threadIdx.x];
        const int a = threadIdx.x / FR_B, b = threadIdx.x % FR_B;
        if (v0 + a < nV && j0 + b < n) scores[(size_t)(j0 + b) * nV + v0 + a] = t;
    }
}

__global__ void __launch_bounds__(256) few_rows_max_kernel(const double* __restrict__ scores, int nV, double* __restrict__ out) {
    __shared__ double sh[8];
    __shared__ int snan;
    const double* r = scores + (size_t)blockIdx.x * nV;
    if (threadIdx.x == 0) snan = 0;
    __syncthreads();
    double m = -INFINITY;
    for (int v = threadIdx.x; v < nV; v += 256) {
        const double x = r[v];
        if (x != x) snan = 1;
        m = fmax(m, x);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = -INFINITY;
        for (int w = 0; w < 8; w++) t = fmax(t, sh[w]);
        out[blockIdx.x] = snan ? __longlong_as_double(0x7ff8000000000000ll) : t;
    }
}

struct HsviOut {
    double best_a, best_o, max_qv, best_v_diff;
    long long added, key0, key1, n_possible;
};

// The decisions of one level (one block).  Stored beliefs return their stored value (keys of the successors against the stored keys);
// Q-values and the observation choice in the reference's order and arithmetic (strict >, so the first maximiser wins; observations of
// probability zero are skipped: their successor is 0/0); append of (key(b), Q) when the recursion continues and b is not stored yet.
__global__ void __launch_bounds__(256) hsvi_choose_kernel(const double* __restrict__ mass, const double* __restrict__ upperSaw, const double* __restrict__ lower,
                                                          const unsigned long long* __restrict__ succKeys, const unsigned long long* __restrict__ bKey,
                                                          const double* __restrict__ rb, unsigned long long* __restrict__ storedKeys,
                                                          double* __restrict__ storedVals, int nStored, int storedCap, int A, int O, double gamma,
                                                          double convTerm, int mayContinue, HsviOut* __restrict__ out) {
    extern __shared__ double s_upper[];      // [A*O]
    __shared__ int s_found;
    const int nZ = A * O;
    for (int z = threadIdx.x; z < nZ; z += 256) s_upper[z] = upperSaw[z];
    if (threadIdx.x == 0) s_found = 0;
    __syncthreads();
    const unsigned long long b0 = bKey[0], b1 = bKey[1];
    for (int i = threadIdx.x; i < nStored; i += 256) {
        const unsigned long long k0 = storedKeys[(size_t)i * 2], k1 = storedKeys[(size_t)i * 2 + 1];
        if (k0 == b0 && k1 == b1) s_found = 1;
        for (int z = 0; z < nZ; z++)
            if (succKeys[(size_t)z * 2] == k0 && succKeys[(size_t)z * 2 + 1] == k1) s_upper[z] = storedVals[i];     // keys are unique: one writer
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double maxQ = -INFINITY;
    int bestA = -1, nPossible = 0;
    for (int a = 0; a < A; a++) {
        double acc = 0.0;
        for (int o = 0; o < O; o++) {
            const double p = mass[a * O + o];
            if (p > 0.0) { acc = __dadd_rn(acc, __dmul_rn(p, s_upper[a * O + o])); nPossible++; }
        }
        const double q = __dadd_rn(rb[a], __dmul_rn(gamma, acc));
        if (q > maxQ) { maxQ = q; bestA = a; }
    }
    double maxOVal = -INFINITY, bestDiff = -INFINITY;
    int bestO = -1;
    if (bestA >= 0)
        for (int o = 0; o < O; o++) {
            const double p = mass[bestA * O + o];
            if (!(p > 0.0)) continue;
            const double diff = __dadd_rn(s_upper[bestA * O + o], -lower[bestA * O + o]);
            const double ov = __dmul_rn(p, diff);
            if (ov > maxOVal) { maxOVal = ov; bestDiff = diff; bestO = o; }
        }
    int added = 0;
    if (mayContinue && !(bestDiff < convTerm) && !s_found && nStored < storedCap) {
        storedKeys[(size_t)nStored * 2] = b0;
        storedKeys[(size_t)nStored * 2 + 1] = b1;
        storedVals[nStored] = maxQ;
        added = 1;
    }
    out->best_a = bestA; out->best_o = bestO; out->max_qv = maxQ; out->best_v_diff = bestDiff;
    out->added = added; out->key0 = (long long)b0; out->key1 = (long long)b1; out->n_possible = nPossible;
}

// next[s] = the chosen successor (b itself when no observation is possible), picked with the indices the choose kernel left on the device
__global__ void __launch_bounds__(256) hsvi_take_next_kernel(const double* __restrict__ succ, const double* __restrict__ b, const HsviOut* __restrict__ res,
                                                             int O, int S, double* __restrict__ next) {
    const int s = blockIdx.x * 256 + threadIdx.x;
    if (s >= S) return;
    const int a = (int)res->best_a, o = (int)res->best_o;
    next[s] = (a >= 0 && o >= 0) ? succ[((size_t)a * O + o) * S + s] : b[s];
}

// ---- point-based upper-bound backup over a slab of beliefs (pbvi_upper_backup) -----------------------------------------------------
// rb[i][a] = b_i . Rbar[:,a]: reward_dot_kernel with a warp per (belief, action)
__global__ void __launch_bounds__(256) reward_dots_kernel(const double* __restrict__ b, int n, int S, const int32_t* __restrict__ nzPtr,
                                                          const int32_t* __restrict__ nzIdx, const double* __restrict__ nzVal, int A,
                                                          double* __restrict__ rb) {
    const int w = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n * A) return;
    const int i = w / A, a = w - i * A;
    const double* bi = b + (size_t)i * S;
    double part = 0.0;
    for (int j = nzPtr[a] + lane; j < nzPtr[a + 1]; j += 32) part = fma(bi[nzIdx[j]], nzVal[j], part);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) part += __shfl_down_sync(0xffffffffu, part, off);
    if (lane == 0) rb[w] = part;
}

// Thread per belief i:  u[i] = max_a [ rb[i][a] + gamma * sum_{o: P(o|b,a) > 0} P(o|b,a) * min(fib, saw)(b^{ao}) ]  (o ascending, products
// and sums rounded one at a time, strict > so the first maximising action wins), cur[i] = min(fib, saw)(b_i), bestA[i] = that action.
// Observations of probability zero are skipped: their successor is the 0/0 row.
__global__ void __launch_bounds__(128) upper_q_kernel(const double* __restrict__ mass, const double* __restrict__ fibSucc,
                                                      const double* __restrict__ sawSucc, const double* __restrict__ rb,
                                                      const double* __restrict__ fibB, const double* __restrict__ sawB, int n, int A, int O,
                                                      double gamma, double* __restrict__ u, double* __restrict__ cur, int32_t* __restrict__ bestA) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n) return;
    const size_t z0 = (size_t)i * A * O;
    double maxQ = -INFINITY;
    int best = -1;
    for (int a = 0; a < A; a++) {
        double acc = 0.0;
        for (int o = 0; o < O; o++) {
            const size_t z = z0 + (size_t)a * O + o;
            const double p = mass[z];
            if (p > 0.0) acc = __dadd_rn(acc, __dmul_rn(p, fmin(fibSucc[z], sawSucc[z])));
        }
        const double q = __dadd_rn(rb[(size_t)i * A + a], __dmul_rn(gamma, acc));
        if (q > maxQ) { maxQ = q; best = a; }
    }
    u[i] = maxQ;
    if (cur) cur[i] = fmin(fibB[i], sawB[i]);
    if (bestA) bestA[i] = best;
}

// out[j] = max_v rows[j] . alphas[v] for any number of rows (few_rows_scores_kernel's grid is limited to 65535 row tiles per launch)
static int few_rows_max_impl(pbvi_model* m, const double* d_rows, int n, const double* d_alphas, int nV, double* d_out, cudaStream_t st) {
    PBVI_TAKE(scores, double, (size_t)n * nV);
    constexpr int SLAB = 65535 * FR_B;
    for (int j0 = 0; j0 < n; j0 += SLAB) {
        const int nj = std::min(SLAB, n - j0);
        few_rows_scores_kernel<<<dim3(ceil_div(nV, FR_A), ceil_div(nj, FR_B)), 256, 0, st>>>(d_rows + (size_t)j0 * m->S, nj, d_alphas, nV, m->S,
                                                                                         scores + (size_t)j0 * nV);
        m->last_launches++;
    }
    few_rows_max_kernel<<<n, 256, 0, st>>>(scores, nV, d_out);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

}  // namespace pbvi

using namespace pbvi;

extern "C" int pbvi_support_lists(pbvi_model* m, const double* d_rows, int n, const double* d_corner, int32_t* d_idx, double* d_val,
                                  int32_t* d_count, double* d_dot, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n >= 0, "n must be non-negative");
    if (n == 0) return PBVI_OK;
    PBVI_REQUIRE(d_rows && d_corner && d_idx && d_val && d_count && d_dot, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    support_lists_kernel<<<n, 256, 0, (cudaStream_t)stream>>>(d_rows, d_corner, m->S, d_idx, d_val, d_count, d_dot);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

namespace pbvi {
// upper bounds of n_q query rows over the stored beliefs given as support lists; scratch from the arena (no reset here)
static int sawtooth_lists_impl(pbvi_model* m, const double* d_corner, const int32_t* d_idx, const double* d_val, const int32_t* d_count,
                               const double* d_dot, const double* d_ub_values, int n_ub, const double* d_queries, int n_q,
                               const double* d_query_mass, double* d_out, cudaStream_t st) {
    PBVI_TAKE(terms, double, (size_t)n_q * (n_ub + 1));
    PBVI_TAKE(v0, double, (size_t)n_q);
    sawtooth_v0_terms_kernel<<<n_q, 256, 0, st>>>(d_corner, d_queries, m->S, n_ub, v0, terms);
    if (n_ub > 0)
        sawtooth_lists_kernel<<<n_ub, 256, 0, st>>>(d_idx, d_val, d_count, d_dot, d_ub_values, n_ub, d_queries, n_q, m->S, v0, d_query_mass, terms);
    row_min_lists_kernel<<<ceil_div(n_q, 128), 128, 0, st>>>(terms, n_q, n_ub + 1, d_out);
    m->last_launches += 3;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}
}  // namespace pbvi

extern "C" int pbvi_sawtooth_lists(pbvi_model* m, const double* d_corner, const int32_t* d_idx, const double* d_val, const int32_t* d_count,
                                   const double* d_dot, const double* d_ub_values, int n_ub, const double* d_queries, int n_q, double* d_out,
                                   void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n_ub >= 0 && n_q >= 0, "counts must be non-negative");
    if (n_q == 0) return PBVI_OK;
    PBVI_REQUIRE(d_corner && d_queries && d_out && (n_ub == 0 || (d_idx && d_val && d_count && d_dot && d_ub_values)), "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    m->last_launches = 0;
    return sawtooth_lists_impl(m, d_corner, d_idx, d_val, d_count, d_dot, d_ub_values, n_ub, d_queries, n_q, nullptr, d_out, (cudaStream_t)stream);
}

extern "C" int pbvi_hsvi_level(pbvi_model* m, const double* d_b, const double* d_alphas, int nV, double gamma, const double* d_corner,
                               const int32_t* d_idx, const double* d_val, const int32_t* d_count, const double* d_dot,
                               const double* d_ub_values, int n_ub, uint64_t* d_stored_keys, double* d_stored_vals, int n_stored,
                               int stored_capacity, double conv_term, int may_continue, double* d_next, double* d_succ, double* d_mass,
                               double* h_out8, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(d_b && d_alphas && d_corner && h_out8, "NULL pointer argument");
    PBVI_REQUIRE(nV > 0 && n_ub >= 0 && n_stored >= 0 && stored_capacity >= n_stored, "bad counts");
    PBVI_REQUIRE(n_ub == 0 || (d_idx && d_val && d_count && d_dot && d_ub_values), "support lists are required when n_ub > 0");
    PBVI_REQUIRE(n_stored == 0 || stored_capacity == 0 || (d_stored_keys && d_stored_vals), "stored key / value arrays are required");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    m->last_launches = 0;
    const int nZ = m->nZ, S = m->S;
    PBVI_TAKE(keys, unsigned long long, (size_t)(nZ + 1) * 2);          // successors, then b itself
    PBVI_TAKE(upper, double, (size_t)nZ);
    PBVI_TAKE(lower, double, (size_t)nZ);
    PBVI_TAKE(rb, double, (size_t)m->A);
    PBVI_TAKE(outDev, HsviOut, 1);
    if (!d_succ) { d_succ = m->arena.take<double>((size_t)nZ * S); if (!d_succ) return PBVI_ERR_OOM; }     // the caller does not want the block
    if (!d_mass) { d_mass = m->arena.take<double>((size_t)nZ); if (!d_mass) return PBVI_ERR_OOM; }
    PBVI_TRY(belief_successors_impl(m, d_b, 1, 1, d_succ, d_mass, st));
    PBVI_TRY(row_hash_launch(m, d_succ, nZ, S, reinterpret_cast<uint64_t*>(keys), st));
    PBVI_TRY(row_hash_launch(m, d_b, 1, S, reinterpret_cast<uint64_t*>(keys + (size_t)nZ * 2), st));
    PBVI_TRY(sawtooth_lists_impl(m, d_corner, d_idx, d_val, d_count, d_dot, d_ub_values, n_ub, d_succ, nZ, d_mass, upper, st));
    reward_dot_kernel<<<ceil_div(m->A * 32, 256), 256, 0, st>>>(d_b, m->rbarNzPtr, m->rbarNzIdx, m->rbarNzVal, m->A, rb);
    m->last_launches++;
    PBVI_TAKE(scores, double, (size_t)nZ * nV);
    few_rows_scores_kernel<<<dim3(ceil_div(nV, FR_A), ceil_div(nZ, FR_B)), 256, 0, st>>>(d_succ, nZ, d_alphas, nV, S, scores);
    few_rows_max_kernel<<<nZ, 256, 0, st>>>(scores, nV, lower);
    m->last_launches += 2;
    hsvi_choose_kernel<<<1, 256, (size_t)nZ * sizeof(double), st>>>(d_mass, upper, lower, keys, keys + (size_t)nZ * 2, rb,
                                                                    reinterpret_cast<unsigned long long*>(d_stored_keys), d_stored_vals, n_stored,
                                                                    stored_capacity, m->A, m->O, gamma, conv_term, may_continue, outDev);
    m->last_launches++;
    if (d_next) {
        hsvi_take_next_kernel<<<ceil_div(S, 256), 256, 0, st>>>(d_succ, d_b, outDev, m->O, S, d_next);
        m->last_launches++;
    }
    PBVI_CUDA(cudaGetLastError());
    PBVI_CUDA(cudaMemcpyAsync(h_out8, outDev, sizeof(HsviOut), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    return PBVI_OK;
}

extern "C" int pbvi_upper_backup(pbvi_model* m, const double* d_b, int n, const double* d_fib, int k, double gamma, const double* d_corner,
                                 const int32_t* d_idx, const double* d_val, const int32_t* d_count, const double* d_dot,
                                 const double* d_ub_values, int n_ub, double* d_u, double* d_cur, int32_t* d_best_a, void* stream) {
    PBVI_REQUIRE(n >= 0 && n_ub >= 0 && k > 0, "counts must be non-negative and k positive");
    if (n > 0) {
        PBVI_REQUIRE(d_b && d_fib && d_corner && d_u, "NULL pointer argument");
        PBVI_REQUIRE(n_ub == 0 || (d_idx && d_val && d_count && d_dot && d_ub_values), "NULL pointer argument: support lists are required when n_ub > 0");
    }
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    if (n == 0) return PBVI_OK;
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, st));
    m->last_launches = 0;
    const int A = m->A, O = m->O, S = m->S;
    const size_t nZ = (size_t)n * m->nZ;
    PBVI_REQUIRE(nZ <= (size_t)INT32_MAX, "too many successors in one call: pass fewer beliefs");
    PBVI_TAKE(succ, double, nZ * S);
    PBVI_TAKE(mass, double, nZ);
    PBVI_TAKE(fibSucc, double, nZ);
    PBVI_TAKE(sawSucc, double, nZ);
    PBVI_TAKE(rb, double, (size_t)n * A);
    PBVI_TAKE(fibB, double, (size_t)n);
    PBVI_TAKE(sawB, double, (size_t)n);
    PBVI_TRY(belief_successors_impl(m, d_b, n, 1, succ, mass, st));
    PBVI_TRY(few_rows_max_impl(m, succ, (int)nZ, d_fib, k, fibSucc, st));
    PBVI_TRY(sawtooth_lists_impl(m, d_corner, d_idx, d_val, d_count, d_dot, d_ub_values, n_ub, succ, (int)nZ, mass, sawSucc, st));
    reward_dots_kernel<<<ceil_div(n * A, 8), 256, 0, st>>>(d_b, n, S, m->rbarNzPtr, m->rbarNzIdx, m->rbarNzVal, A, rb);
    m->last_launches++;
    if (d_cur) {
        PBVI_TRY(few_rows_max_impl(m, d_b, n, d_fib, k, fibB, st));
        PBVI_TRY(sawtooth_lists_impl(m, d_corner, d_idx, d_val, d_count, d_dot, d_ub_values, n_ub, d_b, n, nullptr, sawB, st));
    }
    upper_q_kernel<<<ceil_div(n, 128), 128, 0, st>>>(mass, fibSucc, sawSucc, rb, fibB, sawB, n, A, O, gamma, d_u, d_cur, d_best_a);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

// ---- one level of K gap-driven trials (pbvi_gap_trial_step) ---------------------------------------------------------------------
namespace pbvi {
// rows[k*O + o] = the successor b_k^{a*_k o} (block per row); zeros for an impossible observation, whose successor is the 0/0 row: the
// lower bounds of these rows go through the score kernel, and a NaN row would switch its zero-skipping off for the whole call
__global__ void __launch_bounds__(256) gap_gather_kernel(const double* __restrict__ succ, const double* __restrict__ mass,
                                                         const int32_t* __restrict__ bestA, int O, int nZ, int S, double* __restrict__ rows) {
    const int r = blockIdx.x;
    const int k = r / O, o = r - k * O, a = bestA[k];
    const size_t z = (size_t)k * nZ + (size_t)max(a, 0) * O + o;
    const bool live = a >= 0 && mass[z] > 0.0;
    const double* src = succ + z * S;
    double* dst = rows + (size_t)r * S;
    for (int s = threadIdx.x; s < S; s += 256) dst[s] = live ? src[s] : 0.0;
}

// e_o = P_o * ((U_o - L_o) - theta), one rounding per operation; a NaN excess counts as not positive
__device__ __forceinline__ double gap_excess(double p, double u, double l, double theta) {
    return __dmul_rn(p, __dadd_rn(__dadd_rn(u, -l), -theta));
}

// Thread per trial k: the excess of every possible observation of a*_k and the choice of o*_k.  Without a uniform (or u_k < 0) the
// first maximiser of e over {e > 0}; otherwise o ~ e over that set by NumPy's rule (w = max(e, 0) over all o, cdf = cumsum(w) with
// sequential adds, cdf /= cdf[-1], searchsorted(cdf, u, 'right')), capped at the last positive weight so that a uniform outside [0, 1)
// cannot pick an observation of weight 0.  No positive excess: o*_k = -1.  out4[k] = {a*, o*, Q*, e_{o*}}; with o* = -1, e is the
// largest excess of a possible observation (-inf when there is none).
__global__ void __launch_bounds__(128) gap_choose_kernel(const double* __restrict__ mass, const double* __restrict__ fibSucc,
                                                         const double* __restrict__ sawSucc, const double* __restrict__ lower,
                                                         const int32_t* __restrict__ bestA, const double* __restrict__ q, int K, int A, int O,
                                                         double theta, const double* __restrict__ uniform, double* __restrict__ out4,
                                                         int32_t* __restrict__ bestO, double* __restrict__ uOut, double* __restrict__ lOut) {
    const int k = blockIdx.x * 128 + threadIdx.x;
    if (k >= K) return;
    const int a = bestA[k];                 // -1 only when every Q is NaN: no observation is possible then
    const size_t z0 = (size_t)k * A * O + (size_t)max(a, 0) * O;
    double best = 0.0, top = -INFINITY, tot = 0.0;
    int arg = -1, lastPos = -1;
    for (int o = 0; o < O; o++) {
        const double p = a >= 0 ? mass[z0 + o] : 0.0;
        double u = __longlong_as_double(0x7ff8000000000000ll), l = u;
        if (p > 0.0) {
            u = fmin(fibSucc[z0 + o], sawSucc[z0 + o]);
            l = lower[(size_t)k * O + o];
            const double e = gap_excess(p, u, l, theta);
            top = fmax(top, e);
            if (e > best) { best = e; arg = o; }
            if (e > 0.0) { tot = __dadd_rn(tot, e); lastPos = o; }
        }
        if (uOut) { uOut[(size_t)k * O + o] = u; lOut[(size_t)k * O + o] = l; }
    }
    double eStar = top;
    if (arg >= 0) {
        eStar = best;
        const double uk = uniform ? uniform[k] : -1.0;
        if (uk >= 0.0) {
            double run = 0.0;
            int idx = 0;
            for (int o = 0; o < O; o++) {
                const double p = mass[z0 + o];
                if (p > 0.0) {
                    const double e = gap_excess(p, fmin(fibSucc[z0 + o], sawSucc[z0 + o]), lower[(size_t)k * O + o], theta);
                    if (e > 0.0) run = __dadd_rn(run, e);
                }
                if (__ddiv_rn(run, tot) <= uk) idx++;
            }
            arg = min(idx, lastPos);
            eStar = gap_excess(mass[z0 + arg], fmin(fibSucc[z0 + arg], sawSucc[z0 + arg]), lower[(size_t)k * O + arg], theta);
        }
    }
    out4[(size_t)k * 4 + 0] = a;
    out4[(size_t)k * 4 + 1] = arg;
    out4[(size_t)k * 4 + 2] = q[k];
    out4[(size_t)k * 4 + 3] = eStar;
    bestO[k] = arg;
}

// next[k] = b_k^{a*_k o*_k}, the row pbvi_belief_update(b_k, a*_k, o*_k, normalise = 1) gives (same projection and pairwise normaliser);
// b_k itself when the trial ends (o*_k = -1).  Block per trial.
__global__ void __launch_bounds__(256) gap_next_kernel(const double* __restrict__ succ, const double* __restrict__ b,
                                                       const int32_t* __restrict__ bestA, const int32_t* __restrict__ bestO, int O, int nZ,
                                                       int S, double* __restrict__ next) {
    const int k = blockIdx.x;
    const int o = bestO[k];
    const double* src = o >= 0 ? succ + ((size_t)k * nZ + (size_t)bestA[k] * O + o) * S : b + (size_t)k * S;
    double* dst = next + (size_t)k * S;
    for (int s = threadIdx.x; s < S; s += 256) dst[s] = src[s];
}
}  // namespace pbvi

extern "C" int pbvi_gap_trial_step(pbvi_model* m, const double* d_b, int K, const double* d_lower, int N, const double* d_fib, int k,
                                   double gamma, const double* d_corner, const int32_t* d_idx, const double* d_val, const int32_t* d_count,
                                   const double* d_dot, const double* d_ub_values, int n_ub, double theta, const double* d_uniform,
                                   double* d_out4, double* d_next, double* d_U, double* d_L, void* stream) {
    PBVI_REQUIRE(K >= 0 && n_ub >= 0, "counts must be non-negative");
    PBVI_REQUIRE(N >= 1 && k >= 1, "N >= 1 lower rows and k >= 1 FIB rows are required");
    PBVI_REQUIRE(theta == theta, "theta is NaN");
    PBVI_REQUIRE((d_U == nullptr) == (d_L == nullptr), "d_U and d_L go together");
    if (K > 0) {
        PBVI_REQUIRE(d_b && d_lower && d_fib && d_corner && d_out4 && d_next, "NULL pointer argument");
        PBVI_REQUIRE(n_ub == 0 || (d_idx && d_val && d_count && d_dot && d_ub_values), "NULL pointer argument: support lists are required when n_ub > 0");
    }
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    if (K == 0) return PBVI_OK;
    const int A = m->A, O = m->O, S = m->S;
    const size_t nZ = (size_t)K * m->nZ;
    PBVI_REQUIRE(nZ <= (size_t)INT32_MAX, "too many successors in one call: pass fewer trials");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, st));
    m->last_launches = 0;
    PBVI_TAKE(succ, double, nZ * S);
    PBVI_TAKE(mass, double, nZ);
    PBVI_TAKE(fibSucc, double, nZ);
    PBVI_TAKE(sawSucc, double, nZ);
    PBVI_TAKE(rb, double, (size_t)K * A);
    PBVI_TAKE(q, double, (size_t)K);
    PBVI_TAKE(bestA, int32_t, (size_t)K);
    PBVI_TAKE(bestO, int32_t, (size_t)K);
    PBVI_TAKE(rows, double, (size_t)K * O * S);
    PBVI_TAKE(lower, double, (size_t)K * O);
    // Q and a* exactly as pbvi_upper_backup computes them (same launches on the same inputs)
    PBVI_TRY(belief_successors_impl(m, d_b, K, 1, succ, mass, st));
    PBVI_TRY(few_rows_max_impl(m, succ, (int)nZ, d_fib, k, fibSucc, st));
    PBVI_TRY(sawtooth_lists_impl(m, d_corner, d_idx, d_val, d_count, d_dot, d_ub_values, n_ub, succ, (int)nZ, mass, sawSucc, st));
    reward_dots_kernel<<<ceil_div(K * A, 8), 256, 0, st>>>(d_b, K, S, m->rbarNzPtr, m->rbarNzIdx, m->rbarNzVal, A, rb);
    upper_q_kernel<<<ceil_div(K, 128), 128, 0, st>>>(mass, fibSucc, sawSucc, rb, nullptr, nullptr, K, A, O, gamma, q, nullptr, bestA);
    // L_o = max_n X_n . b^{a* o} for the O successors of a* only
    gap_gather_kernel<<<K * O, 256, 0, st>>>(succ, mass, bestA, O, m->nZ, S, rows);
    m->last_launches += 3;
    PBVI_TRY(max_values_impl(m, rows, K * O, d_lower, N, lower, nullptr, st));
    gap_choose_kernel<<<ceil_div(K, 128), 128, 0, st>>>(mass, fibSucc, sawSucc, lower, bestA, q, K, A, O, theta, d_uniform, d_out4, bestO,
                                                        d_U, d_L);
    gap_next_kernel<<<K, 256, 0, st>>>(succ, d_b, bestA, bestO, O, m->nZ, S, d_next);
    m->last_launches += 2;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}
