// Set semantics on raw bytes (reference src/mdp.py:668-669, 773-774; src/pomdp.py:581, 600), the MDP value-iteration
// sweep (src/mdp.py:1507), pointwise-domination pruning (src/mdp.py:857-866), HSVI's sawtooth upper bound
// (src/pomdp.py:887-895) and SSEA's novelty distance (src/pomdp.py:1682-1686).  All HBM-bound streaming kernels.
#include <algorithm>

#include <cub/device/device_radix_sort.cuh>

#include "pbvi_common.cuh"

namespace pbvi {

// 128-bit key of the raw 8-byte words of each row (NH hashes with position keys, pbvi_common.cuh).  Block per row.
__global__ void __launch_bounds__(256) row_hash_kernel(const uint64_t* __restrict__ rows, int rowLen, uint64_t* __restrict__ out) {
    __shared__ uint64_t sh[2][8];
    const uint64_t* row = rows + (size_t)blockIdx.x * rowLen;
    uint64_t h0 = 0, h1 = 0;
    for (int i = threadIdx.x; i < rowLen; i += 256) {
        const uint64_t w = row[i];
        const uint4 k = row_key_words(i);
        h0 += row_hash_term0(w, k);
        h1 += row_hash_term1(w, k);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        h0 += __shfl_down_sync(0xffffffffu, h0, off);
        h1 += __shfl_down_sync(0xffffffffu, h1, off);
    }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = h0; sh[1][threadIdx.x >> 5] = h1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t a = 0, b = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) { a += sh[0][w]; b += sh[1][w]; }
        out[(size_t)blockIdx.x * 2] = row_hash_final0(a, rowLen);
        out[(size_t)blockIdx.x * 2 + 1] = row_hash_final1(b, rowLen);
    }
}

__global__ void __launch_bounds__(256) rows_equal_kernel(const uint64_t* __restrict__ ra, const int32_t* __restrict__ ia,
                                                         const uint64_t* __restrict__ rb, const int32_t* __restrict__ ib, int rowLen,
                                                         int32_t* __restrict__ flags) {
    const uint64_t* a = ra + (size_t)ia[blockIdx.x] * rowLen;
    const uint64_t* b = rb + (size_t)ib[blockIdx.x] * rowLen;
    int diff = 0;
    for (int i = threadIdx.x; i < rowLen; i += 256) diff |= (a[i] != b[i]);
    const int any = __syncthreads_or(diff);
    if (threadIdx.x == 0) flags[blockIdx.x] = any ? 0 : 1;
}

// ---- first-occurrence grouping of fixed-width keys: the insertion order of a Python dict (src/mdp.py:668-669, src/pomdp.py:600)
//      computed on the device, so the (a*, v*) tuples of a backup and the 128-bit keys of its rows never travel to the host.
//      Open-addressing table of representatives; per slot an atomicMin of the record index (first position) and an atomicMax of
//      (rank << 32 | index) (the record that defines the group's action: last occurrence, or largest caller-supplied rank).
//      Which record becomes the representative of a slot depends on scheduling; first / last / inverse do not.
__device__ __forceinline__ uint32_t key_hash(const uint32_t* __restrict__ k, int w) {
    uint64_t h = 0x9e3779b97f4a7c15ull;
    for (int j = 0; j < w; j++) h = mix64(h ^ (uint64_t)k[j]) + 0xd6e8feb86659fd93ull;
    return (uint32_t)(h >> 29);
}

__global__ void __launch_bounds__(256) group_init_kernel(int32_t* __restrict__ rep, int32_t* __restrict__ gfirst,
                                                         unsigned long long* __restrict__ glast, int T) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= T) return;
    rep[i] = -1;
    gfirst[i] = 0x7fffffff;
    glast[i] = 0ull;
}

__global__ void __launch_bounds__(256) group_insert_kernel(const uint32_t* __restrict__ keys, int n, int w, const int32_t* __restrict__ rank,
                                                           int T, int32_t* rep, int32_t* __restrict__ gfirst,
                                                           unsigned long long* __restrict__ glast, int32_t* __restrict__ slotOf) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const uint32_t* k = keys + (size_t)i * w;
    uint32_t h = key_hash(k, w) & (uint32_t)(T - 1);
    for (;;) {
        int cur = *reinterpret_cast<volatile int32_t*>(rep + h);
        if (cur == -1) {
            cur = atomicCAS(rep + h, -1, i);
            if (cur == -1) break;                       // this record now represents the slot
        }
        const uint32_t* kc = keys + (size_t)cur * w;
        bool eq = true;
        for (int j = 0; j < w; j++) eq &= (kc[j] == k[j]);
        if (eq) break;
        h = (h + 1) & (uint32_t)(T - 1);
    }
    slotOf[i] = (int32_t)h;
    atomicMin(gfirst + h, i);
    atomicMax(glast + h, ((unsigned long long)(uint32_t)(rank ? rank[i] : i) << 32) | (unsigned long long)(uint32_t)i);
}

// The same insertion over the all-gathered blocks of the sharded backup's tuple exchange: `world` blocks of blockRows rows of
// (w + 2) int32 words; row 0 of a block is its header (word 0 = number of records u_r), rows 1..u_r are records
// (key[w], first position, last position).  Positions are positions in the WHOLE belief set, so the merge does not depend on how
// the beliefs are spread over the ranks (contiguous blocks, or the append-only interleaved ownership of the sharded solve): a
// group's first record is the one with the smallest first position, its last record the one with the largest last position, and
// the groups come out ordered by their first position (group_collect_kernel + a radix sort of the (position, row) words).
// maxCount receives max_r u_r (overflow check of the caller).
__global__ void __launch_bounds__(256) group_insert_blocks_kernel(const int32_t* __restrict__ blocks, int world, int blockRows, int w, int T,
                                                                  int32_t* rep, unsigned long long* __restrict__ gfirst,
                                                                  unsigned long long* __restrict__ glast, int32_t* __restrict__ maxCount) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= world * blockRows) return;
    const int stride = w + 2;
    const int r = i / blockRows, j = i - r * blockRows;
    const int count = blocks[(size_t)r * blockRows * stride];
    if (j == 0) atomicMax(maxCount, count);
    if (j == 0 || j > count) return;
    const uint32_t* k = reinterpret_cast<const uint32_t*>(blocks) + (size_t)i * stride;
    uint32_t h = key_hash(k, w) & (uint32_t)(T - 1);
    for (;;) {
        int cur = *reinterpret_cast<volatile int32_t*>(rep + h);
        if (cur == -1) {
            cur = atomicCAS(rep + h, -1, i);
            if (cur == -1) break;
        }
        const uint32_t* kc = reinterpret_cast<const uint32_t*>(blocks) + (size_t)cur * stride;
        bool eq = true;
        for (int x = 0; x < w; x++) eq &= (kc[x] == k[x]);
        if (eq) break;
        h = (h + 1) & (uint32_t)(T - 1);
    }
    atomicMin(gfirst + h, ((unsigned long long)k[w] << 32) | (unsigned long long)(uint32_t)i);
    atomicMax(glast + h, ((unsigned long long)k[w + 1] << 32) | (unsigned long long)(uint32_t)i);
}

__global__ void __launch_bounds__(256) group_blocks_init_kernel(int32_t* __restrict__ rep, unsigned long long* __restrict__ gfirst,
                                                                unsigned long long* __restrict__ glast, int T,
                                                                unsigned long long* __restrict__ sortKeys, int n) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < T) { rep[i] = -1; gfirst[i] = ~0ull; glast[i] = 0ull; }
    if (i < n) sortKeys[i] = ~0ull;                    // unused sort slots sink to the end
}

// occupied slots -> (first position << 32 | row of that record, slot), unordered; count[0] = number of groups
__global__ void __launch_bounds__(256) group_collect_kernel(const int32_t* __restrict__ rep, const unsigned long long* __restrict__ gfirst, int T,
                                                            unsigned long long* __restrict__ sortKeys, int32_t* __restrict__ sortSlots,
                                                            int32_t* __restrict__ count) {
    const int h = blockIdx.x * 256 + threadIdx.x;
    const bool used = h < T && rep[h] != -1;
    const unsigned bal = __ballot_sync(0xffffffffu, used);
    int base = 0;
    if ((threadIdx.x & 31) == 0 && bal) base = atomicAdd(count, __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (used) {
        const int at = base + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u));
        sortKeys[at] = gfirst[h];
        sortSlots[at] = h;
    }
}

__global__ void __launch_bounds__(256) group_emit_kernel(const unsigned long long* __restrict__ sortedKeys, const int32_t* __restrict__ sortedSlots,
                                                         const unsigned long long* __restrict__ glast, const int32_t* __restrict__ count,
                                                         int32_t* __restrict__ first, int32_t* __restrict__ last) {
    const int g = blockIdx.x * 256 + threadIdx.x;
    if (g >= *count) return;
    first[g] = (int32_t)(sortedKeys[g] & 0xffffffffull);
    last[g] = (int32_t)(glast[sortedSlots[g]] & 0xffffffffull);
}

// one block: stream compaction of the group-first records in ascending index order (tiles of 1024, ballot scan)
__global__ void __launch_bounds__(1024) group_compact_kernel(const int32_t* __restrict__ slotOf, const int32_t* __restrict__ gfirst,
                                                             const unsigned long long* __restrict__ glast, int n,
                                                             int32_t* __restrict__ groupOfSlot, int32_t* __restrict__ first,
                                                             int32_t* __restrict__ last, int32_t* __restrict__ count) {
    __shared__ int warpCount[32];
    __shared__ int base;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) base = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += 1024) {
        const int i = i0 + tid;
        int slot = 0;
        bool isFirst = false;
        if (i < n) {
            slot = slotOf[i];
            isFirst = slot >= 0 && gfirst[slot] == i;       // slot < 0: not a record (header / padding row of a gathered block)
        }
        const unsigned bal = __ballot_sync(0xffffffffu, isFirst);
        if (lane == 0) warpCount[w] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            const int c = warpCount[j];
            before += (j < w) ? c : 0;
            total += c;
        }
        const int b0 = base;
        if (isFirst) {
            const int g = b0 + before + __popc(bal & ((1u << lane) - 1u));
            first[g] = i;
            last[g] = (int32_t)(glast[slot] & 0xffffffffull);
            groupOfSlot[slot] = g;
        }
        __syncthreads();
        if (tid == 0) base = b0 + total;
        __syncthreads();
    }
    if (tid == 0) *count = base;
}

__global__ void __launch_bounds__(256) group_inverse_kernel(const int32_t* __restrict__ slotOf, const int32_t* __restrict__ groupOfSlot, int n,
                                                            int32_t* __restrict__ inverse) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < n) inverse[i] = groupOfSlot[slotOf[i]];
}

// block per record: a record that is not the first of its group must equal that first row bytewise (confirms the 128-bit key match)
__global__ void __launch_bounds__(256) group_confirm_kernel(const uint64_t* __restrict__ rows, int rowLen, const int32_t* __restrict__ first,
                                                            const int32_t* __restrict__ inverse, int32_t* __restrict__ mismatch) {
    const int i = blockIdx.x, f = first[inverse[i]];
    if (f == i) return;
    const uint64_t* a = rows + (size_t)i * rowLen;
    const uint64_t* b = rows + (size_t)f * rowLen;
    int diff = 0;
    for (int s = threadIdx.x; s < rowLen; s += 256) diff |= (a[s] != b[s]);
    if (diff) atomicOr(mismatch, 1);
}

// alpha[a][s] = Rbar[s,a] + gamma * sum_r P[s,a,r] * V*[reach[s,a,r]]; vopt_out[s] = max_a
__global__ void __launch_bounds__(256) vi_sweep_kernel(const double* __restrict__ vopt, const int32_t* __restrict__ reachK,
                                                       const double* __restrict__ probK, const double* __restrict__ rbarT, double gamma,
                                                       int S, int R, int A, double* __restrict__ alphaOut, double* __restrict__ voptOut) {
    const int s = blockIdx.x * 256 + threadIdx.x;
    if (s >= S) return;
    double best = -INFINITY;
    for (int a = 0; a < A; a++) {
        const size_t base = ((size_t)a * S + s) * R;
        double inner = 0.0;
        for (int r = 0; r < R; r++) {
            const double prod = __dmul_rn(probK[base + r], vopt[reachK[base + r]]);
            inner = (r == 0) ? prod : __dadd_rn(inner, prod);
        }
        const double v = __dadd_rn(rbarT[(size_t)a * S + s], __dmul_rn(gamma, inner));
        if (alphaOut) alphaOut[(size_t)a * S + s] = v;
        best = fmax(best, v);
    }
    if (voptOut) voptOut[s] = best;
}

// Fast Informed Bound sweep (Hauskrecht 2000), thread per (a, s):
//     out[a][s] = Rbar[s,a] + gamma * sum_o max_{a' < k} sum_r RTO[s,a,o,r] * U[a'][reach[s,a,r]]
// U is read through its transposed copy UT [S][k], so the k candidates of one landing state are contiguous.  Fixed order: r ascending
// inside, then o ascending, products and sums rounded one at a time (no fma) as in vi_sweep_kernel -- R = 1 models reproduce a NumPy
// restatement bit for bit.  With stats != nullptr (k == A, rows paired by index) every block also leaves max(out - U) and max |out - U|
// (NaN wins) in part[block]; the last block to finish reduces the parts in block order into stats[2].
constexpr int FIB_THREADS = 256;

__global__ void __launch_bounds__(FIB_THREADS) fib_sweep_kernel(const double* __restrict__ UT, int k, const int32_t* __restrict__ reachK,
                                                                const double* __restrict__ rtoK, const double* __restrict__ rbarT, double gamma,
                                                                int S, int R, int A, int O, double* __restrict__ out,
                                                                double2* __restrict__ part, unsigned int* __restrict__ done,
                                                                double* __restrict__ stats) {
    __shared__ double sh[2][FIB_THREADS / 32];
    __shared__ bool s_last;
    const int t = blockIdx.x * FIB_THREADS + threadIdx.x;
    double dmax = -INFINITY, amax = 0.0;
    bool nan = false;
    if (t < A * S) {
        const int a = t / S, s = t - a * S;
        const size_t K = (size_t)S * R;
        const size_t base = (size_t)s * R;
        const int32_t* reach = reachK + (size_t)a * K + base;
        double acc = 0.0;
        for (int o = 0; o < O; o++) {
            const double* rto = rtoK + ((size_t)a * O + o) * K + base;
            double best = -INFINITY;
            for (int ap = 0; ap < k; ap++) {
                double inner = 0.0;
                for (int r = 0; r < R; r++) {
                    const double prod = __dmul_rn(rto[r], UT[(size_t)reach[r] * k + ap]);
                    inner = (r == 0) ? prod : __dadd_rn(inner, prod);
                }
                best = (inner != inner || best != best) ? inner + best : fmax(best, inner);     // NaN wins (np.max)
            }
            acc = __dadd_rn(acc, best);
        }
        const double v = __dadd_rn(rbarT[(size_t)a * S + s], __dmul_rn(gamma, acc));
        out[(size_t)a * S + s] = v;
        if (stats) {
            const double d = __dadd_rn(v, -UT[(size_t)s * k + a]);
            nan = d != d;
            dmax = d;
            amax = fabs(d);
        }
    }
    if (!stats) return;
    // block reduction (NaN wins), then the last-block reduction of the per-block parts
    const unsigned anyNan = __ballot_sync(0xffffffffu, nan);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        dmax = fmax(dmax, __shfl_down_sync(0xffffffffu, dmax, off));
        amax = fmax(amax, __shfl_down_sync(0xffffffffu, amax, off));
    }
    if ((threadIdx.x & 31) == 0) {
        sh[0][threadIdx.x >> 5] = anyNan ? NAN : dmax;
        sh[1][threadIdx.x >> 5] = anyNan ? NAN : amax;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double m0 = -INFINITY, m1 = 0.0;
        bool bn = false;
        for (int w = 0; w < FIB_THREADS / 32; w++) {
            bn |= sh[0][w] != sh[0][w];
            m0 = fmax(m0, sh[0][w]);
            m1 = fmax(m1, sh[1][w]);
        }
        part[blockIdx.x] = bn ? make_double2(NAN, NAN) : make_double2(m0, m1);
        __threadfence();
        s_last = atomicAdd(done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        const volatile double* pv = reinterpret_cast<volatile double*>(part);     // written by other blocks: bypass L1
        double m0 = -INFINITY, m1 = 0.0;
        bool bn = false;
        for (int b = 0; b < (int)gridDim.x; b++) {
            const double x = pv[2 * b], y = pv[2 * b + 1];
            bn |= x != x;
            m0 = fmax(m0, x);
            m1 = fmax(m1, y);
        }
        stats[0] = bn ? NAN : m0;
        stats[1] = bn ? NAN : m1;
    }
}

// keep[i] = 1 iff exactly one vector (alpha_i itself, or none when it holds a NaN... the reference counts rows with
// all(alpha_j >= alpha_i)) dominates alpha_i everywhere.  Block per i, early exit per j on the first losing coordinate block.
__global__ void __launch_bounds__(256) prune_dominated_kernel(const double* __restrict__ alphas, int nV, int S, int32_t* __restrict__ keep) {
    const int i = blockIdx.x;
    const double* ai = alphas + (size_t)i * S;
    int count = 0;
    for (int j = 0; j < nV; j++) {
        const double* aj = alphas + (size_t)j * S;
        int dominated = 1;
        for (int s0 = 0; s0 < S && dominated; s0 += 256 * 8) {
            int ok = 1;
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int s = s0 + u * 256 + threadIdx.x;
                if (s < S && !(aj[s] >= ai[s])) ok = 0;
            }
            dominated = __syncthreads_and(ok);
        }
        count += dominated;
    }
    if (threadIdx.x == 0) keep[i] = (count == 1) ? 1 : 0;
}

// first[i] = the smallest j with Y_j[s] >= X_i[s] at every state (a NaN on either side is a violation), or -1.  Block per (32 old rows
// x 32 new rows) tile; both tiles pass through shared memory DOM_KS states at a time, and each thread carries four (j, i) pairs, i =
// lane, j = warp + 8 q, so a warp reads one broadcast Y value and 32 consecutive X values per state.  A pair drops out at its first
// violating state and the block stops when none is left.  first[] starts at -1 (all ones) and the tiles meet through an unsigned
// atomicMin, so the result does not depend on the order of the blocks; a pair whose j is not below the best j already found for its i is
// dropped at the start.
// kSelf (pbvi_dominating_row: Y and X are the same rows): the pair j = i is excluded, and a pair with j > i also has to be strictly greater
// at some state ("above" collects that bit per pair), so that of two equal rows only the later one has a witness.
constexpr int DOM_T = 32, DOM_KS = 32;

template <bool kSelf>
__global__ void __launch_bounds__(256) first_dominating_row_kernel(const double* __restrict__ Y, int nNew, const double* __restrict__ X, int nOld,
                                                                   int S, int32_t* first) {
    __shared__ double xs[DOM_KS][DOM_T + 1], ys[DOM_KS][DOM_T + 1];
    const int i0 = blockIdx.x * DOM_T, j0 = blockIdx.y * DOM_T;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = i0 + lane;
    const unsigned best = (i < nOld) ? *(volatile unsigned*)(first + i) : 0u;
    unsigned alive = 0, above = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int j = j0 + warp + 8 * q;
        if (i < nOld && j < nNew && (unsigned)j < best && (!kSelf || j != i)) alive |= 1u << q;
    }
    for (int s0 = 0; s0 < S; s0 += DOM_KS) {
        if (!__syncthreads_or(alive != 0)) return;                     // also: the tiles of the previous chunk have been read
#pragma unroll
        for (int u = 0; u < DOM_T * DOM_KS / 256; u++) {
            const int r = warp + 8 * u, s = s0 + lane;
            xs[lane][r] = (i0 + r < nOld && s < S) ? X[(size_t)(i0 + r) * S + s] : 0.0;
            ys[lane][r] = (j0 + r < nNew && s < S) ? Y[(size_t)(j0 + r) * S + s] : 0.0;
        }
        __syncthreads();
        const int ks = min(DOM_KS, S - s0);
        for (int c = 0; c < ks && alive; c++) {
            const double x = xs[c][lane];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const double y = ys[c][warp + 8 * q];
                if (!(y >= x)) alive &= ~(1u << q);
                if (kSelf && y > x) above |= 1u << q;
            }
        }
    }
    if (kSelf) {
#pragma unroll
        for (int q = 0; q < 4; q++)
            if (j0 + warp + 8 * q > i && !(above & (1u << q))) alive &= ~(1u << q);
    }
    // the lowest surviving j of this thread, then of the block per i: the atomic keeps the lowest over all tiles
#pragma unroll
    for (int q = 0; q < 4; q++)
        if (alive & (1u << q)) {
            atomicMin((unsigned*)(first + i), (unsigned)(j0 + warp + 8 * q));
            break;
        }
}

// Sawtooth upper bound:  v0_q = q . corner;  terms[q][i] = v0_q + (ub_value_i - ub_belief_i . corner) * min_{s: ub_belief_i[s] > 0} q[s] / ub_belief_i[s];
// terms[q][nUb] = v0_q;  row_min_kernel then takes out[q] = min_i terms[q][i].
// One block per STORED belief i, for all queries: b_i is read from HBM once (the first version, one block per (i, q), re-read
// b_i, the corner values and the query for every pair: 28 GB per HSVI level at 3000 stored beliefs and 18 successors).  The
// support of b_i is compacted, one range of SAW_RANGE states at a time, into shared memory as (state, value) pairs; each query
// then gathers only those states.  Same arithmetic per element (exact division, min is order-free): bit-identical results.
// Measured on the 40-expansion HSVI solve of the olfactory model (tools/solve_olfactory.py): expand 11.1 s -> 9.4 s.  Two other
// forms were tried and are slower there: a warp per query with a reciprocal-screened two-pass minimum (12.2 s) and a dense walk
// with eight query loads in flight per thread (12.9 s); the per-level host round trips now weigh as much as this kernel.
constexpr int SAW_RANGE = 8192;
constexpr int SAW_Q_SLAB = 4096;

__global__ void __launch_bounds__(256) sawtooth_v0_kernel(const double* __restrict__ corner, const double* __restrict__ queries, int S,
                                                          double* __restrict__ v0) {
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
    }
}

__global__ void __launch_bounds__(256) sawtooth_terms_kernel(const double* __restrict__ corner, const double* __restrict__ ubB,
                                                             const double* __restrict__ ubV, int nUb, const double* __restrict__ queries,
                                                             int nQ, int S, const double* __restrict__ v0, double* __restrict__ terms) {
    extern __shared__ __align__(16) unsigned char saw_smem[];
    double* sval = reinterpret_cast<double*>(saw_smem);                       // [SAW_RANGE] b_i values on the support
    int* sidx = reinterpret_cast<int*>(saw_smem + sizeof(double) * SAW_RANGE);   // [SAW_RANGE] their states
    double* sratio = reinterpret_cast<double*>(saw_smem + (sizeof(double) + sizeof(int)) * SAW_RANGE);   // [nQ]
    __shared__ double sh[8];
    __shared__ int scount;
    const int i = blockIdx.x;
    const double* bi = ubB + (size_t)i * S;
    double dotp = 0.0;
    for (int s = threadIdx.x; s < S; s += 256) dotp = fma(bi[s], corner[s], dotp);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dotp += __shfl_down_sync(0xffffffffu, dotp, off);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = dotp;
    for (int q = threadIdx.x; q < nQ; q += 256) sratio[q] = INFINITY;
    __syncthreads();
    double d = 0.0;
    for (int w = 0; w < 8; w++) d += sh[w];                                      // every thread: same order as thread 0 of the first version
    for (int s0 = 0; s0 < S; s0 += SAW_RANGE) {
        __syncthreads();
        if (threadIdx.x == 0) scount = 0;
        __syncthreads();
        const int s1 = min(S, s0 + SAW_RANGE);
        for (int s = s0 + threadIdx.x; s < s1; s += 256) {
            const double b = bi[s];
            if (b > 0.0) {
                const int slot = atomicAdd(&scount, 1);
                sval[slot] = b;
                sidx[slot] = s;
            }
        }
        __syncthreads();
        const int cnt = scount;
        if (cnt == 0) continue;
        for (int q = 0; q < nQ; q++) {
            const double* qq = queries + (size_t)q * S;
            double r = INFINITY;
            for (int j = threadIdx.x; j < cnt; j += 256) r = fmin(r, qq[sidx[j]] / sval[j]);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) r = fmin(r, __shfl_down_sync(0xffffffffu, r, off));
            if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = r;
            __syncthreads();
            if (threadIdx.x == 0) {
                double m = sratio[q];
                for (int w = 0; w < 8; w++) m = fmin(m, sh[w]);
                sratio[q] = m;
            }
            __syncthreads();
        }
    }
    __syncthreads();
    for (int q = threadIdx.x; q < nQ; q += 256) terms[(size_t)q * (nUb + 1) + i] = v0[q] + (ubV[i] - d) * sratio[q];
}

__global__ void __launch_bounds__(128) row_min_kernel(const double* __restrict__ terms, int n, int width, double* __restrict__ out) {
    const int qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= n) return;
    double best = INFINITY;
    for (int i = 0; i < width; i++) best = fmin(best, terms[(size_t)qi * width + i]);
    out[qi] = best;
}

// out[j] = min_i || beliefs[i] - candidates[j] ||_2  (SSEA novelty, src/pomdp.py:1682-1686: the reference forms the whole
// [B, B*A*O, S] difference tensor).  Tiled like a GEMM, with the reference's DIRECT arithmetic sum_s (b - c)^2 -- the expanded form
// |b|^2 + |c|^2 - 2 b.c would cancel catastrophically exactly where the distance matters (successors close to the set).  A block owns
// L2_TC candidates and walks all beliefs in tiles of L2_TB; state chunks of L2_TS go through shared memory; a thread accumulates a
// 4 x 4 block of pair sums, so every shared-memory load feeds four subtract-multiply-adds.  np.min propagates NaN (the all-NaN
// successor of an impossible observation): any NaN pair sum makes the candidate's result NaN.
constexpr int L2_TC = 64, L2_TB = 64, L2_TS = 32;

__global__ void __launch_bounds__(256) min_l2_tiled_kernel(const double* __restrict__ beliefs, int nB, const double* __restrict__ cands, int nC,
                                                           int S, double* __restrict__ out) {
    __shared__ double sc[L2_TS][L2_TC + 1];      // [state][candidate]: the four candidates of a thread are 16 apart (no bank conflicts)
    __shared__ double sb[L2_TS][L2_TB + 1];
    __shared__ double smin[16][L2_TC];
    __shared__ int snan[L2_TC];
    const int tid = threadIdx.x, tc = tid & 15, tb = tid >> 4;     // candidate lane / belief lane of the 16 x 16 thread grid
    const int c0 = blockIdx.x * L2_TC;
    double best[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
    bool sawNan[4] = {false, false, false, false};
    for (int b0 = 0; b0 < nB; b0 += L2_TB) {
        double acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) acc[i][j] = 0.0;
        for (int s0 = 0; s0 < S; s0 += L2_TS) {
            __syncthreads();
            // 64 rows x 32 states per tile, 256 threads: thread loads rows r = tid / 32 + 8 k at state tid % 32 (coalesced)
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int r = (tid >> 5) + 8 * k, sx = tid & 31, s = s0 + sx;
                sc[sx][r] = (c0 + r < nC && s < S) ? cands[(size_t)(c0 + r) * S + s] : 0.0;
                sb[sx][r] = (b0 + r < nB && s < S) ? beliefs[(size_t)(b0 + r) * S + s] : 0.0;
            }
            __syncthreads();
#pragma unroll 8
            for (int sx = 0; sx < L2_TS; sx++) {
                double cv[4], bv[4];
#pragma unroll
                for (int i = 0; i < 4; i++) { cv[i] = sc[sx][tc + 16 * i]; bv[i] = sb[sx][tb + 16 * i]; }
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) { const double d = bv[j] - cv[i]; acc[i][j] = fma(d, d, acc[i][j]); }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (b0 + tb + 16 * j < nB) {
                    if (acc[i][j] != acc[i][j]) sawNan[i] = true;
                    best[i] = fmin(best[i], acc[i][j]);
                }
    }
    __syncthreads();
    if (tid < L2_TC) snan[tid] = 0;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; i++) {
        smin[tb][tc + 16 * i] = best[i];
        if (sawNan[i]) snan[tc + 16 * i] = 1;
    }
    __syncthreads();
    if (tid < L2_TC && c0 + tid < nC) {
        double m = INFINITY;
#pragma unroll
        for (int k = 0; k < 16; k++) m = fmin(m, smin[k][tid]);
        out[c0 + tid] = snan[tid] ? NAN : sqrt(m);
    }
}

// GER error term of one successor (block per (b, z)): sum_s (alpha'[s] - alpha_b[s]) * (succ[s] - b[s]),
// alpha'[s] = r_max where the successor gained mass, r_min elsewhere (src/pomdp.py:1738-1748).
// A NaN successor (impossible observation) yields 0: its weight P(o|b,a) is 0.
__global__ void __launch_bounds__(256) ger_eps_kernel(const double* __restrict__ beliefs, const double* __restrict__ alphaB,
                                                      const double* __restrict__ succ, int S, int nZ, double rMin, double rMax,
                                                      double* __restrict__ eps) {
    __shared__ double sh[8];
    const int z = blockIdx.x, b = blockIdx.y;
    const double* bel = beliefs + (size_t)b * S;
    const double* al = alphaB + (size_t)b * S;
    const double* sc = succ + ((size_t)b * nZ + z) * S;
    double part = 0.0;
    for (int s = threadIdx.x; s < S; s += 256) {
        const double d = sc[s] - bel[s];
        part = fma((d >= 0.0 ? rMax : rMin) - al[s], d, part);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) part += __shfl_down_sync(0xffffffffu, part, off);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; w++) t += sh[w];
        eps[(size_t)b * nZ + z] = (t != t) ? 0.0 : t;
    }
}

int row_hash_launch(pbvi_model* m, const double* d_rows, int n, int row_len, uint64_t* d_hash, cudaStream_t st) {
    row_hash_kernel<<<n, 256, 0, st>>>(reinterpret_cast<const uint64_t*>(d_rows), row_len, d_hash);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

int configure_misc_kernels() {
    PBVI_CUDA(cudaFuncSetAttribute(sawtooth_terms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)((sizeof(double) + sizeof(int)) * SAW_RANGE + sizeof(double) * SAW_Q_SLAB)));
    return PBVI_OK;
}

}  // namespace pbvi

using namespace pbvi;

extern "C" int pbvi_ger_scores(pbvi_model* m, const double* d_beliefs, const double* d_alpha_b, const double* d_succ, int n,
                               double r_min, double r_max, double* d_eps, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n >= 0, "n must be non-negative");
    if (n == 0) return PBVI_OK;
    PBVI_REQUIRE(d_beliefs && d_alpha_b && d_succ && d_eps, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    for (int i0 = 0; i0 < n; i0 += 65535) {
        const int ni = std::min(65535, n - i0);
        ger_eps_kernel<<<dim3(m->nZ, ni), 256, 0, (cudaStream_t)stream>>>(d_beliefs + (size_t)i0 * m->S, d_alpha_b + (size_t)i0 * m->S,
                                                                         d_succ + (size_t)i0 * m->nZ * m->S, m->S, m->nZ, r_min, r_max,
                                                                         d_eps + (size_t)i0 * m->nZ);
    }
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_row_hash(pbvi_model* m, const double* d_rows, int n, int row_len, uint64_t* d_hash, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n >= 0 && row_len > 0, "need n >= 0 rows of positive length");
    if (n == 0) return PBVI_OK;
    PBVI_REQUIRE(d_rows && d_hash, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    row_hash_kernel<<<n, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint64_t*>(d_rows), row_len, d_hash);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_rows_equal(pbvi_model* m, const double* d_rows_a, const int32_t* d_ia, const double* d_rows_b, const int32_t* d_ib,
                               int n, int row_len, int32_t* d_flags, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n >= 0 && row_len > 0, "need n >= 0 pairs of positive length");
    if (n == 0) return PBVI_OK;
    PBVI_REQUIRE(d_rows_a && d_rows_b && d_ia && d_ib && d_flags, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    rows_equal_kernel<<<n, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint64_t*>(d_rows_a), d_ia,
                                                          reinterpret_cast<const uint64_t*>(d_rows_b), d_ib, row_len, d_flags);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

namespace pbvi {
// First-occurrence grouping of n records of `words` 32-bit words (see pbvi_group_keys); scratch from the arena, nothing read back:
// *d_count_out points at the group count on the device.
int group_keys_impl(pbvi_model* m, const uint32_t* d_keys, int n, int words, const int32_t* d_rank, int32_t* d_first, int32_t* d_last,
                    int32_t* d_inverse, int32_t** d_count_out, cudaStream_t st) {
    int T = 64;
    while (T < 2 * n) T <<= 1;
    PBVI_TAKE(rep, int32_t, (size_t)T);
    PBVI_TAKE(gfirst, int32_t, (size_t)T);
    PBVI_TAKE(glast, unsigned long long, (size_t)T);
    PBVI_TAKE(slotOf, int32_t, (size_t)n);
    PBVI_TAKE(groupOfSlot, int32_t, (size_t)T);
    PBVI_TAKE(count, int32_t, 1);
    group_init_kernel<<<ceil_div(T, 256), 256, 0, st>>>(rep, gfirst, glast, T);
    group_insert_kernel<<<ceil_div(n, 256), 256, 0, st>>>(d_keys, n, words, d_rank, T, rep, gfirst, glast, slotOf);
    group_compact_kernel<<<1, 1024, 0, st>>>(slotOf, gfirst, glast, n, groupOfSlot, d_first, d_last, count);
    m->last_launches += 3;
    if (d_inverse) {
        group_inverse_kernel<<<ceil_div(n, 256), 256, 0, st>>>(slotOf, groupOfSlot, n, d_inverse);
        m->last_launches++;
    }
    PBVI_CUDA(cudaGetLastError());
    *d_count_out = count;
    return PBVI_OK;
}

// mismatch[0] != 0 afterwards iff some row differs bytewise from the first row of its group
int confirm_groups_launch(pbvi_model* m, const double* d_rows, int n, int row_len, const int32_t* d_first, const int32_t* d_inverse,
                          int32_t* d_mismatch, cudaStream_t st) {
    PBVI_CUDA(cudaMemsetAsync(d_mismatch, 0, sizeof(int32_t), st));
    group_confirm_kernel<<<n, 256, 0, st>>>(reinterpret_cast<const uint64_t*>(d_rows), row_len, d_first, d_inverse, d_mismatch);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}
}  // namespace pbvi

extern "C" int pbvi_group_keys(pbvi_model* m, const uint32_t* d_keys, int n, int words, const int32_t* d_rank, int32_t* d_first,
                               int32_t* d_last, int32_t* d_inverse, int* h_count, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n >= 0 && words > 0 && h_count != nullptr, "need n >= 0 records of positive width and a count output");
    *h_count = 0;
    m->last_launches = 0;
    if (n == 0) return PBVI_OK;
    PBVI_REQUIRE(d_keys && d_first && d_last, "NULL pointer argument");
    PBVI_REQUIRE(n <= (1 << 29), "too many records");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    int32_t* count = nullptr;
    PBVI_TRY(group_keys_impl(m, d_keys, n, words, d_rank, d_first, d_last, d_inverse, &count, st));
    int32_t c = 0;
    PBVI_CUDA(cudaMemcpyAsync(&c, count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    *h_count = (int)c;
    return PBVI_OK;
}

extern "C" int pbvi_group_record_blocks(pbvi_model* m, const int32_t* d_blocks, int world, int block_rows, int words, int32_t* d_first,
                                       int32_t* d_last, int* h_count, int* h_max_records, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(world > 0 && block_rows > 1 && words > 0 && h_count && h_max_records, "need world > 0 blocks of more than one row");
    PBVI_REQUIRE(d_blocks && d_first && d_last, "NULL pointer argument");
    const long long n = (long long)world * block_rows;
    PBVI_REQUIRE(n <= (1 << 29), "too many records");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    int T = 64;
    while (T < 2 * n) T <<= 1;
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    PBVI_TAKE(rep, int32_t, (size_t)T);
    PBVI_TAKE(gfirst, unsigned long long, (size_t)T);
    PBVI_TAKE(glast, unsigned long long, (size_t)T);
    PBVI_TAKE(keysIn, unsigned long long, (size_t)n);
    PBVI_TAKE(keysOut, unsigned long long, (size_t)n);
    PBVI_TAKE(slotsIn, int32_t, (size_t)n);
    PBVI_TAKE(slotsOut, int32_t, (size_t)n);
    PBVI_TAKE(count, int32_t, 2);
    size_t sortBytes = 0;
    PBVI_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, keysIn, keysOut, slotsIn, slotsOut, (int)n, 0, 64, st));
    PBVI_TAKE(sortTemp, char, sortBytes);
    PBVI_CUDA(cudaMemsetAsync(count, 0, 2 * sizeof(int32_t), st));
    group_blocks_init_kernel<<<ceil_div(std::max<int>(T, (int)n), 256), 256, 0, st>>>(rep, gfirst, glast, T, keysIn, (int)n);
    group_insert_blocks_kernel<<<ceil_div((int)n, 256), 256, 0, st>>>(d_blocks, world, block_rows, words, T, rep, gfirst, glast, count + 1);
    group_collect_kernel<<<ceil_div(T, 256), 256, 0, st>>>(rep, gfirst, T, keysIn, slotsIn, count);
    PBVI_CUDA(cub::DeviceRadixSort::SortPairs(sortTemp, sortBytes, keysIn, keysOut, slotsIn, slotsOut, (int)n, 0, 64, st));
    group_emit_kernel<<<ceil_div((int)n, 256), 256, 0, st>>>(keysOut, slotsOut, glast, count, d_first, d_last);
    m->last_launches = 5;
    PBVI_CUDA(cudaGetLastError());
    int32_t c[2] = {0, 0};
    PBVI_CUDA(cudaMemcpyAsync(c, count, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    *h_count = (int)c[0];
    *h_max_records = (int)c[1];
    return PBVI_OK;
}

extern "C" int pbvi_confirm_groups(pbvi_model* m, const double* d_rows, int n, int row_len, const int32_t* d_first, const int32_t* d_inverse,
                                   int* h_all_equal, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n >= 0 && row_len > 0 && h_all_equal != nullptr, "need n >= 0 rows of positive length and a result output");
    *h_all_equal = 1;
    m->last_launches = 0;
    if (n == 0) return PBVI_OK;
    PBVI_REQUIRE(d_rows && d_first && d_inverse, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    PBVI_TAKE(mismatch, int32_t, 1);
    PBVI_TRY(confirm_groups_launch(m, d_rows, n, row_len, d_first, d_inverse, mismatch, st));
    int32_t bad = 0;
    PBVI_CUDA(cudaMemcpyAsync(&bad, mismatch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    *h_all_equal = bad ? 0 : 1;
    return PBVI_OK;
}

extern "C" int pbvi_vi_sweep(pbvi_model* m, const double* d_vopt, double gamma, double* d_alpha_out, double* d_vopt_out, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(d_vopt != nullptr, "vopt pointer is NULL");
    if (!m->has_probs) {
        set_error("the model was created without reachable_probabilities; the VI sweep is unavailable");
        return PBVI_ERR_UNSUPPORTED;
    }
    PBVI_CUDA(cudaSetDevice(m->device));
    vi_sweep_kernel<<<ceil_div(m->S, 256), 256, 0, (cudaStream_t)stream>>>(d_vopt, m->reachK, m->probK, m->rbarT, gamma, m->S, m->R, m->A,
                                                                          d_alpha_out, d_vopt_out);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_fib_sweep(pbvi_model* m, const double* d_in, int k, double gamma, double* d_out, double* d_stats2, void* stream) {
    PBVI_REQUIRE(k > 0, "k must be positive");
    PBVI_REQUIRE(d_in && d_out, "NULL pointer argument");
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(!d_stats2 || k == m->A, "the residual statistics pair rows by index: they need k == A input rows");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, st));
    m->last_launches = 0;
    const int S = m->S, nBlocks = ceil_div(m->A * S, FIB_THREADS);
    PBVI_TAKE(UT, double, (size_t)S * k);
    PBVI_TRY(transpose_alphas(m, d_in, k, k, UT, st));          // [k][S] -> [S][k]: the k candidates of a landing state are one line
    double2* part = nullptr;
    unsigned int* done = nullptr;
    if (d_stats2) {
        part = m->arena.take<double2>((size_t)nBlocks);
        done = m->arena.take<unsigned int>(1);
        if (!part || !done) return PBVI_ERR_OOM;
        PBVI_CUDA(cudaMemsetAsync(done, 0, sizeof(unsigned int), st));
    }
    fib_sweep_kernel<<<nBlocks, FIB_THREADS, 0, st>>>(UT, k, m->reachK, m->rtoK, m->rbarT, gamma, S, m->R, m->A, m->O, d_out, part, done, d_stats2);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_prune_dominated(pbvi_model* m, const double* d_alphas, int nV, int32_t* d_keep, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(nV >= 0, "nV must be non-negative");
    if (nV == 0) return PBVI_OK;
    PBVI_REQUIRE(d_alphas && d_keep, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    prune_dominated_kernel<<<nV, 256, 0, (cudaStream_t)stream>>>(d_alphas, nV, m->S, d_keep);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_first_dominating_row(pbvi_model* m, const double* d_new, int n_new, const double* d_old, int n_old, int32_t* d_first,
                                         void* stream) {
    PBVI_REQUIRE(n_new >= 0 && n_old >= 0, "n_new and n_old must be non-negative");
    PBVI_REQUIRE(n_old == 0 || (d_old && d_first && (n_new == 0 || d_new)), "NULL pointer argument");
    PBVI_REQUIRE(n_new <= 65535 * DOM_T, "n_new above 65535 * 32 (grid.y)");
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    if (n_old == 0) return PBVI_OK;
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_CUDA(cudaMemsetAsync(d_first, 0xFF, (size_t)n_old * sizeof(int32_t), st));
    m->last_launches = 0;
    if (n_new == 0) return PBVI_OK;
    first_dominating_row_kernel<false><<<dim3(ceil_div(n_old, DOM_T), ceil_div(n_new, DOM_T)), 256, 0, st>>>(d_new, n_new, d_old, n_old, m->S,
                                                                                                             d_first);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_dominating_row(pbvi_model* m, const double* d_rows, int n, int32_t* d_witness, void* stream) {
    PBVI_REQUIRE(n >= 0, "n must be non-negative");
    PBVI_REQUIRE(n == 0 || (d_rows && d_witness), "NULL pointer argument");
    PBVI_REQUIRE(n <= 65535 * DOM_T, "n above 65535 * 32 (grid.y)");
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    m->last_launches = 0;
    if (n == 0) return PBVI_OK;
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_CUDA(cudaMemsetAsync(d_witness, 0xFF, (size_t)n * sizeof(int32_t), st));
    first_dominating_row_kernel<true><<<dim3(ceil_div(n, DOM_T), ceil_div(n, DOM_T)), 256, 0, st>>>(d_rows, n, d_rows, n, m->S, d_witness);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_sawtooth(pbvi_model* m, const double* d_corner, const double* d_ub_beliefs, const double* d_ub_values, int n_ub,
                             const double* d_queries, int n_q, double* d_out, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n_ub >= 0 && n_q >= 0, "counts must be non-negative");
    if (n_q == 0) return PBVI_OK;
    PBVI_REQUIRE(d_corner && d_queries && d_out && (n_ub == 0 || (d_ub_beliefs && d_ub_values)), "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    PBVI_TAKE(terms, double, (size_t)n_q * (n_ub + 1));
    // column n_ub of `terms` holds v0_q itself (the corner term of the minimum); the stored-belief blocks read it from there
    PBVI_TAKE(v0, double, (size_t)n_q);
    cudaStream_t st = (cudaStream_t)stream;
    sawtooth_v0_kernel<<<n_q, 256, 0, st>>>(d_corner, d_queries, m->S, v0);
    m->last_launches = 1;
    PBVI_CUDA(cudaMemcpy2DAsync(terms + n_ub, (size_t)(n_ub + 1) * sizeof(double), v0, sizeof(double), sizeof(double), (size_t)n_q,
                                cudaMemcpyDeviceToDevice, st));
    if (n_ub > 0) {
        constexpr int Q_SLAB = SAW_Q_SLAB;             // queries per launch (their running minima live in shared memory)
        for (int q0 = 0; q0 < n_q; q0 += Q_SLAB) {
            const int nq = std::min(Q_SLAB, n_q - q0);
            const size_t smem = (sizeof(double) + sizeof(int)) * SAW_RANGE + sizeof(double) * (size_t)nq;
            sawtooth_terms_kernel<<<n_ub, 256, smem, st>>>(d_corner, d_ub_beliefs, d_ub_values, n_ub, d_queries + (size_t)q0 * m->S, nq, m->S,
                                                           v0 + q0, terms + (size_t)q0 * (n_ub + 1));
            m->last_launches++;
        }
    }
    row_min_kernel<<<ceil_div(n_q, 128), 128, 0, (cudaStream_t)stream>>>(terms, n_q, n_ub + 1, d_out);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_min_l2_distance(pbvi_model* m, const double* d_beliefs, int nB, const double* d_candidates, int nC, double* d_out,
                                    void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(nB > 0 && nC >= 0, "need nB > 0 beliefs and nC >= 0 candidates");
    if (nC == 0) return PBVI_OK;
    PBVI_REQUIRE(d_beliefs && d_candidates && d_out, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    min_l2_tiled_kernel<<<ceil_div(nC, L2_TC), 256, 0, (cudaStream_t)stream>>>(d_beliefs, nB, d_candidates, nC, m->S, d_out);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}
