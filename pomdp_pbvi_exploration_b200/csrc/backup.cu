// Point-based backup (reference PBVI_Solver.backup, src/pomdp.py:1447-1524) and max_v b.alpha_v
// (compute_change src/pomdp.py:2165-2167) on sm_100a.  Gamma[a,o,v,s] is never materialised for
// reachable_state_count == 1 models; see score_kernel.cuh for the dominant kernel.
//
// Pipeline of pbvi_backup_select:
//   transpose_kernel          alphas [V][S] -> alphaT [S][Vp]          (so a gathered successor row is one coalesced line)
//   belief_mask_kernel        row-group occupancy bits of every (belief tile, 4-state chunk) + the belief tiles as shared-memory images
//   alpha_row_mask_kernel, chunk_alpha_mask_kernel   which chunks gather a non-zero row of each 64-alpha column quarter
//   build_chunk_lists_kernel  per (tile, a, o, alpha tile): ordered list of live pipeline stages with per-chunk flag bytes
//   (R > 1) gamma_project_kernel  GammaT[a,o][s][v] = sum_r RTO * alphaT[reach]   (HBM-bound gather)
//   score_kernel              persistent block-sparse DMMA GEMM + fused first-index argmax per 64-alpha column quarter
//   combine_tiles_kernel      argmax across the column quarters of all alpha tiles (ascending, strict >)
//   approx_value_kernel, backup_value_kernel   value[b][a] = b . (Rbar[:,a] + sum_o Gamma[a,o,v*]): screened, exact where it matters
//   first_argmax_kernel       a*[b]
// pbvi_backup_assemble:
//   action_order_kernel + assemble_grouped_kernel (R = 1) / assemble_kernel   alpha_a rows for (action, v*[O]) tuples in the
//                             reference's operation order, no FMA contraction, 128-bit row keys accumulated on the way
// pbvi_controller_sweep:
//   controller_sweep_kernel   the same rows for the nodes of a finite-state controller against its own rows, plus a fused residual
// pbvi_controller_evaluate:
//   controller_evaluate_kernel   persistent cooperative launch: the sweeps of controller_sweep_kernel until the change test stops them
#include <algorithm>
#include <thread>

#include <cooperative_groups.h>

#include "score_kernel.cuh"

namespace cg = cooperative_groups;

namespace pbvi {

constexpr int MASK_COLS = 256;                         // states per belief_mask_kernel block
constexpr int MASK_SLABS = MASK_COLS / 32;             // 32-state slabs (one warp load per row)
constexpr int MASK_CHUNKS = MASK_COLS / KC;            // chunks per block
static_assert(NRG == 4 && RG == 16 && 32 % KC == 0 && MASK_SLABS % 2 == 0, "belief_mask_kernel: 8 warps = 4 row groups x 2 slab phases");
static_assert(BN == 256 && NCW == 4, "alpha_row_mask_kernel: four 64-column quarters per alpha tile");

// ---- alphas [V][S] -> alphaT [S][Vp], zero in the pad columns ---------------------------------------------------
__global__ void __launch_bounds__(256) transpose_kernel(const double* __restrict__ in, int V, int S, int Vp, double* __restrict__ out) {
    __shared__ double tile[32][33];
    const int v0 = blockIdx.x * 32, s0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const int v = v0 + ty + j * 8, s = s0 + tx;
        tile[ty + j * 8][tx] = (v < V && s < S) ? in[(size_t)v * S + s] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const int s = s0 + ty + j * 8, v = v0 + tx;
        if (s < S && v < Vp) out[(size_t)s * Vp + v] = tile[tx][ty + j * 8];
    }
}

int transpose_alphas(pbvi_model* m, const double* d_alphas, int nV, int Vp, double* d_alphaT, cudaStream_t st) {
    dim3 grid(ceil_div(Vp, 32), ceil_div(m->S, 32));
    transpose_kernel<<<grid, 256, 0, st>>>(d_alphas, nV, m->S, Vp, d_alphaT);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

// ---- bits[mt][c]: bit g set iff some belief of row group g of tile mt is non-zero on chunk c.  The same pass writes
//      beliefsP, the belief tiles re-laid out as the shared-memory image the score kernel wants:
//          beliefsP[mt][chunk][row group][RG rows][KC]      (columns of row r XOR-swizzled by a_swizzle(r); zero beyond nB rows / S)
//      so that the A operand of one (tile, chunk, row group) is ONE contiguous, 128-byte aligned block of RG*KC doubles that a
//      single bulk async copy drops into shared memory already in its bank-conflict-free layout.  Images of row groups that
//      are all-zero on a chunk are NOT written (the score kernel never fetches them): on the bench workload that is 60 % of
//      the image.  A warp owns one row group and a 32-state slab at a time: 16 independent row loads in flight per lane.
//      Non-finite input (np.argmax / NaN semantics of the reference): a row that holds a NaN or an infinity makes every one of its
//      scores NaN in the reference (NaN * 0 = NaN), so it is only flagged here (rowBad) and combine_tiles_kernel writes the
//      reference's result for it -- v* = 0, score NaN -- whatever the kernel accumulated.  Non-finite ALPHAS (signs[SIGN_DENSE], set
//      by alpha_row_mask_kernel, which runs first) make every zero-skipping rule invalid (0 * inf = NaN): then every row group of
//      every chunk is written and marked live and the score kernel runs the dense product.
__global__ void __launch_bounds__(256) belief_mask_kernel(const double* __restrict__ beliefs, int nB, int S, int nChunks,
                                                          uint8_t* __restrict__ bits, double* __restrict__ beliefsP, int* __restrict__ signs,
                                                          uint8_t* __restrict__ rowBad) {
    __shared__ unsigned smask[MASK_CHUNKS];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int cb = blockIdx.x, mt = blockIdx.y;
    const int rg = w & 3;
    if (tid < MASK_CHUNKS) smask[tid] = 0u;
    __syncthreads();
    const bool dense = signs[SIGN_DENSE] != 0;
    bool bad = false;
    const int row0 = mt * BM + rg * RG;
    constexpr int CPS = 32 / KC;                         // chunks per slab
    for (int sl = (w >> 2); sl < MASK_SLABS; sl += 2) {
        const int s = cb * MASK_COLS + sl * 32 + lane;
        double v[RG];
#pragma unroll
        for (int r = 0; r < RG; r++) v[r] = (row0 + r < nB && s < S) ? beliefs[(size_t)(row0 + r) * S + s] : 0.0;
        bool nz = false;
#pragma unroll
        for (int r = 0; r < RG; r++) {
            nz |= v[r] != 0.0;
            bad |= !(v[r] >= 0.0);                       // negative or NaN entry: no exact-zero shortcut for this call
            if (!(fabs(v[r]) <= 1.79769313486231570e308)) rowBad[row0 + r] = 1;     // NaN / inf (never a pad row: those read 0.0)
        }
        const unsigned bal = __ballot_sync(0xffffffffu, nz);
        const int cl = lane / KC;                        // this lane's chunk inside the slab
        const bool live = dense || ((bal >> (cl * KC)) & ((1u << KC) - 1u)) != 0u;
        const int c = (cb * MASK_COLS + sl * 32) / KC + cl;
        if (live && c < nChunks) {
            double* dst = beliefsP + (((size_t)mt * nChunks + c) * NRG + rg) * A_GROUP_DOUBLES;
            const int col = lane % KC;
#pragma unroll
            for (int r = 0; r < RG; r++) dst[r * KC + (col ^ a_swizzle(r))] = v[r];
            if (col == 0) atomicOr(&smask[sl * CPS + cl], 1u << rg);
        }
    }
    if (bad) signs[1] = 1;
    __syncthreads();
    if (tid < MASK_CHUNKS) {
        const int c = cb * MASK_CHUNKS + tid;
        if (c < nChunks) bits[(size_t)mt * nChunks + c] = (uint8_t)smask[tid];
    }
}

// ---- rowLive[nt][s]: bit q set iff alphaT[s][nt*BN + q*64 .. + 64) holds a non-zero: an all-zero piece of a row of the B operand
//      (an alpha tile that vanishes at a landing state -- the rule for value functions of goal-reward models, whose support
//      grows by one step per backup) contributes exact zeros to every score.  Warp per (s, nt).
__global__ void __launch_bounds__(256) alpha_row_mask_kernel(const double* __restrict__ alphaT, int S, int Vp, int nNt,
                                                             uint8_t* __restrict__ rowLive, int* __restrict__ signs) {
    const size_t gw = ((size_t)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (gw >= (size_t)S * nNt) return;
    const int lane = threadIdx.x & 31;
    const int s = (int)(gw / nNt), nt = (int)(gw % nNt);
    const double* row = alphaT + (size_t)s * Vp + (size_t)nt * BN;
    bool neg = false, nonfinite = false;
    unsigned live = 0u;
#pragma unroll
    for (int j = 0; j < BN / 32; j++) {
        const double v = row[j * 32 + lane];
        neg |= !(v >= 0.0);
        nonfinite |= !(fabs(v) <= 1.79769313486231570e308);
        if (__ballot_sync(0xffffffffu, v != 0.0)) live |= 1u << (j / 2);      // columns j*32 .. j*32+31 lie in quarter j / 2
    }
    if (lane == 0) rowLive[(size_t)nt * S + s] = (uint8_t)live;
    if (neg) signs[0] = 1;
    if (nonfinite) signs[SIGN_DENSE] = 1;
}

// ---- bLive[nt][g][c]: bit q set iff some state k of chunk c gathers an alphaT row that is live in column quarter q: row index
//      reach[g][k] (g = action) for the gather path, k itself when reach == nullptr (plain path, one group)
__global__ void __launch_bounds__(256) chunk_alpha_mask_kernel(const uint8_t* __restrict__ rowLive, const int32_t* __restrict__ reachP,
                                                               int S, int Sp, int nChunks, int nG, int nNt, uint8_t* __restrict__ bLive,
                                                               const int* __restrict__ signs) {
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= (size_t)nNt * nG * nChunks) return;
    if (signs[SIGN_DENSE]) { bLive[i] = 0xFu; return; }          // non-finite alphas: nothing may be skipped
    const int c = (int)(i % nChunks), g = (int)((i / nChunks) % nG), nt = (int)(i / ((size_t)nChunks * nG));
    const uint8_t* live = rowLive + (size_t)nt * S;
    unsigned any = 0;
#pragma unroll
    for (int kk = 0; kk < KC; kk++) {
        const int k = c * KC + kk;
        if (k < S) any |= live[reachP ? reachP[(size_t)g * Sp + k] : k];
    }
    bLive[i] = (uint8_t)any;
}

// ---- ordered list of the live pipeline stages (SUB consecutive chunks) of every (tile, z, alpha tile); one warp per list.  A
//      chunk is live iff some belief of the tile is non-zero on it AND RTO[a][o] is non-zero on it AND the alpha tile is non-zero
//      at some state it lands on.  Entry = (stage index, flags): byte h of flags = live row groups | live column quarters << 4
//      of chunk h of the stage (0 when the chunk is dead).
__global__ void __launch_bounds__(32) build_chunk_lists_kernel(const uint8_t* __restrict__ bits, const uint8_t* __restrict__ zMask,
                                                               const uint8_t* __restrict__ bLive, int nG, int zPerG, int nChunks, int nZ,
                                                               int nNt, uint2* __restrict__ lists, int32_t* __restrict__ counts,
                                                               const int* __restrict__ signs) {
    const int z = blockIdx.x / nNt, nt = blockIdx.x % nNt, mt = blockIdx.y, lane = threadIdx.x;
    const size_t slot = ((size_t)mt * nZ + z) * nNt + nt;
    const int nStages = nChunks / SUB;
    uint2* list = lists + slot * nStages;
    const uint8_t* bl = bLive ? bLive + ((size_t)nt * nG + z / zPerG) * nChunks : nullptr;
    if (signs[SIGN_DENSE]) zMask = nullptr;             // non-finite alphas: a zero RTO factor does not make the term zero
    int base = 0;
    for (int s0 = 0; s0 < nStages; s0 += 32) {
        const int sg = s0 + lane;
        unsigned flags = 0u;
        if (sg < nStages) {
#pragma unroll
            for (int h = 0; h < SUB; h++) {
                const int c = sg * SUB + h;
                unsigned b = bits[(size_t)mt * nChunks + c], q = 0xFu;
                if (zMask && !zMask[(size_t)z * nChunks + c]) b = 0u;
                if (bl) q = bl[c];
                if (b && q) flags |= (b | (q << 4)) << (8 * h);
            }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, flags != 0u);
        if (flags) list[base + __popc(bal & ((1u << lane) - 1u))] = make_uint2((unsigned)sg, flags);
        base += __popc(bal);
    }
    if (lane == 0) counts[slot] = base;
}

// ---- argmax across the column quarters of all alpha tiles: ascending column order, strict > keeps the lowest index on ties ----------------------
//      np.argmax semantics (argmax_append): the first NaN wins, an all -inf row yields column 0; a quarter that lies entirely beyond V carries
//      ARG_NONE and is passed over.  Rows flagged non-finite by belief_mask_kernel get the reference's result outright: every score
//      of such a row is NaN there, so v* = 0 and the maximum is NaN.
__global__ void __launch_bounds__(256) combine_tiles_kernel(const double* __restrict__ pval, const int32_t* __restrict__ pidx, int nNt,
                                                            size_t n, int nZ, int nV, const uint8_t* __restrict__ rowBad,
                                                            double* __restrict__ outVal, int32_t* __restrict__ outIdx) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double best = pval[i];
    int idx = pidx[i];
    for (int t = 1; t < nNt; t++) {
        const int id = pidx[(size_t)t * n + i];
        if (id != ARG_NONE) argmax_append(best, idx, pval[(size_t)t * n + i], id);
    }
    if (rowBad[i / (size_t)nZ]) { best = __longlong_as_double(0x7ff8000000000000ll); idx = 0; }
    if (outVal) outVal[i] = best;
    if (outIdx) outIdx[i] = min(max(idx, 0), nV - 1);
}

// ---- R > 1: GammaT[j][s][v] = sum_r RTO[z][s*R+r] * alphaT[reach[a][s*R+r]][v] for z = zOrder[zBegin + j] ----------
__global__ void __launch_bounds__(256) gamma_project_kernel(const double* __restrict__ alphaT, const int32_t* __restrict__ reachK,
                                                            const double* __restrict__ rtoK, const int32_t* __restrict__ zOrder,
                                                            int zBegin, int S, int R, int O, int Vp, double* __restrict__ out,
                                                            const int* __restrict__ signs) {
    const int j = blockIdx.y, z = zOrder[zBegin + j], a = z / O;
    const bool dense = signs[SIGN_DENSE] != 0;          // non-finite alphas: 0 * inf = NaN must survive, like in the reference's einsum
    const int s0 = blockIdx.x * 8;
    const int32_t* reach = reachK + (size_t)a * S * R;
    const double* rto = rtoK + (size_t)z * S * R;
    for (int idx = threadIdx.x; idx < 8 * Vp; idx += 256) {
        const int sl = idx / Vp, v = idx - sl * Vp, s = s0 + sl;
        if (s >= S) break;
        double acc = 0.0;
        for (int r = 0; r < R; r++) {
            const size_t k = (size_t)s * R + r;
            const double w = rto[k];
            if (w != 0.0 || dense) acc += w * alphaT[(size_t)reach[k] * Vp + v];
        }
        out[((size_t)j * (S + 1) + s) * Vp + v] = acc;
    }
}

// fixed-shape block sum (256 threads): shuffle tree inside each warp, then warp 0 lane 0 adds the 8 partials in order
__device__ __forceinline__ double block_sum_256(double v, double* sh) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double tot = 0.0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 0; w < 8; w++) tot += sh[w];
    }
    return tot;   // valid on thread 0
}

// alpha_a[s] of the reference for one (action, v*[O]) tuple: Rbar[s,a] + ((G_0 + G_1) + ...),
// G_o = gamma * sum_r RTO[s,a,o,r] * alpha[v_o][reach[s,a,r]]  (src/pomdp.py:1489-1502), no FMA contraction.
// skipZero: a term whose RTO factor is zero is taken as +0.0 without gathering the alpha value.  With finite alphas and gamma
// the reference's term is +-0.0; the sign of a zero term changes no partial sum that is non-zero and at most the sign of one
// that is zero, and Rbar + (+-0.0) is the same double unless Rbar is -0.0 -- in which case nothing is skipped.  So the
// result is bit-identical while most gathers of a sparse observation model (2 of 3 observations impossible from most states of
// the olfactory model) are never issued.
// Coherent: the alpha rows were written earlier in the same launch (controller_evaluate_kernel), so they are gathered with ld.global.cg
// instead of through the read-only data cache, which is not kept coherent with writes during a launch.
template <bool Coherent = false>
__device__ __forceinline__ double alpha_a_entry(const double* __restrict__ alphas, int S, int R, int O, const int* vsel,
                                                const int32_t* __restrict__ reach, const double* __restrict__ rtoA,
                                                const double* __restrict__ rbarA, double gamma, int s, bool skipZero) {
    const double rb = rbarA[s];
    const bool skip = skipZero && !(rb == 0.0 && signbit(rb));
    double tot = 0.0;
    for (int o = 0; o < O; o++) {
        const double* arow = alphas + (size_t)vsel[o] * S;
        const double* rto = rtoA + (size_t)o * S * R;
        double inner = 0.0;
        for (int r = 0; r < R; r++) {
            const size_t k = (size_t)s * R + r;
            const double w = rto[k];
            const double prod = (skip && w == 0.0) ? 0.0 : __dmul_rn(w, Coherent ? __ldcg(arow + reach[k]) : arow[reach[k]]);
            inner = (r == 0) ? prod : __dadd_rn(inner, prod);
        }
        const double term = __dmul_rn(gamma, inner);
        tot = (o == 0) ? term : __dadd_rn(tot, term);
    }
    return __dadd_rn(rb, tot);
}

// sets *flag when some entry is NaN or +-inf (the zero-skip of the assemble kernels needs finite alphas)
__global__ void __launch_bounds__(256) nonfinite_scan_kernel(const double* __restrict__ x, size_t n, int* __restrict__ flag) {
    bool bad = false;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) bad |= !(fabs(x[i]) <= 1.79769313486231570e308);
    if (bad) *flag = 1;
}

// ---- approx[b][a] = b . Rbar[:,a] + gamma * sum_o max_v score[b,a,o,v]: the same quantity as value[b][a] below, but summed
//      in the score kernel's order.  Warp per (b, a); only the non-zero rewards are touched.
__global__ void __launch_bounds__(256) approx_value_kernel(const double* __restrict__ beliefs, const double* __restrict__ maxscore,
                                                           const int32_t* __restrict__ nzPtr, const int32_t* __restrict__ nzIdx,
                                                           const double* __restrict__ nzVal, double gamma, int S, int A, int O, int nB,
                                                           double* __restrict__ approx) {
    const size_t gw = ((size_t)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (gw >= (size_t)nB * A) return;
    const int lane = threadIdx.x & 31;
    const int b = (int)(gw / A), a = (int)(gw % A);
    const double* brow = beliefs + (size_t)b * S;
    double part = 0.0;
    for (int j = nzPtr[a] + lane; j < nzPtr[a + 1]; j += 32) part = fma(brow[nzIdx[j]], nzVal[j], part);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) part += __shfl_down_sync(0xffffffffu, part, off);
    if (lane == 0) {
        double so = 0.0;
        for (int o = 0; o < O; o++) so += maxscore[gw * O + o];
        approx[gw] = part + gamma * so;
    }
}

// ---- value[b][a] = sum_s b[s] * alpha_a[b,a,s] in the reference's operation order; block per (a, b); only the support of b
//      is visited.  Screening: an action whose approximate value lies below the best approximate value of its belief by more
//      than the two summation orders can differ cannot be the argmax, so it keeps the approximate value and the block exits;
//      every action that could win or tie is evaluated exactly.
__global__ void __launch_bounds__(256) backup_value_kernel(const double* __restrict__ beliefs, const double* __restrict__ alphas,
                                                           const int32_t* __restrict__ vstar, const int32_t* __restrict__ reachK,
                                                           const double* __restrict__ rtoK, const double* __restrict__ rbarT,
                                                           const double* __restrict__ approx, const int* __restrict__ signs, int modelNonneg,
                                                           const uint8_t* __restrict__ bits, int nChunks, int b0, double gamma, int S, int R,
                                                           int A, int O, int nV, int needExact, double relMargin,
                                                           double* __restrict__ value) {
    extern __shared__ int s_vsel[];
    __shared__ double sh[8];
    const int a = blockIdx.x, b = b0 + blockIdx.y;
    // non-finite alphas: the reference's value is NaN / inf arithmetic over EVERY state (0 * inf = NaN), so nothing is screened or skipped
    const bool dense = signs[SIGN_DENSE] != 0;
    // Screening needs a bound on how far the score-order sum can be from the reference-order sum.  With non-negative terms both
    // rounding errors are below n * eps * value, n = S*R*O terms (7.3e-12 relative for the olfactory model), so relMargin =
    // max(1e-10, 4 * n * eps) times |best| separates safely.  With mixed
    // signs the terms can cancel and the error is bounded by n * eps * sum |terms|, which is not known here: every action is
    // then evaluated exactly (small / reward-penalty models: the pass is cheap there).
    const bool nonneg = modelNonneg && !signs[0] && !signs[1];
    if (!dense && nonneg) {
        const double mine = approx[(size_t)b * A + a];
        // every term of the sum is >= 0 (model, beliefs and alphas are non-negative) and the score-order sum is exactly 0:
        // all terms are zero, so the reference-order sum is exactly +0.0 too
        if (mine == 0.0 && gamma > 0.0) {
            if (threadIdx.x == 0) value[(size_t)b * A + a] = 0.0;
            return;
        }
        double best = -INFINITY;
        for (int aa = 0; aa < A; aa++) best = fmax(best, approx[(size_t)b * A + aa]);
        const double margin = relMargin * fabs(best);
        if (!(mine >= best - margin)) {
            if (threadIdx.x == 0) value[(size_t)b * A + a] = mine;
            return;
        }
        // the only action that can win: a* is decided, and when the caller did not ask for the values themselves the exact sum
        // would change nothing (about 70 % of the beliefs of the olfactory workload)
        if (!needExact) {
            int contenders = 0;
            for (int aa = 0; aa < A; aa++) contenders += (approx[(size_t)b * A + aa] >= best - margin) ? 1 : 0;
            if (contenders == 1) {
                if (threadIdx.x == 0) value[(size_t)b * A + a] = mine;
                return;
            }
        }
    }
    for (int o = threadIdx.x; o < O; o += 256) s_vsel[o] = min(max(vstar[((size_t)b * A + a) * O + o], 0), nV - 1);
    __syncthreads();
    const double* brow = beliefs + (size_t)b * S;
    const int32_t* reach = reachK + (size_t)a * S * R;
    const double* rtoA = rtoK + (size_t)a * O * S * R;
    const double* rbarA = rbarT + (size_t)a * S;
    // no zero-term skipping here: the pass is latency-bound (a few support states per thread), and a gather that waits for its RTO
    // factor serialises two dependent loads (measured: 1.22 -> 1.53 ms with the skip)
    const bool skipZero = false;
    double part = 0.0;
    // KC threads per chunk; chunks on which the belief's row group is all-zero (occupancy bits of belief_mask_kernel)
    // are skipped without touching the belief row.  The state -> thread mapping is the same for every action of a belief.
    const uint8_t* live = bits + (size_t)(b / BM) * nChunks;
    const unsigned gbit = 1u << ((b % BM) / RG);
    for (int c = threadIdx.x / KC; c < nChunks; c += 256 / KC) {
        if (!(live[c] & gbit)) continue;                 // (dense mode: belief_mask_kernel marked every chunk live)
        const int s = c * KC + (threadIdx.x % KC);
        if (s >= S) continue;
        const double bs = brow[s];
        if (bs != 0.0 || dense) part = fma(bs, alpha_a_entry(alphas, S, R, O, s_vsel, reach, rtoA, rbarA, gamma, s, skipZero), part);
    }
    const double tot = block_sum_256(part, sh);
    if (threadIdx.x == 0) value[(size_t)b * A + a] = tot;
}

// ---- first index of the maximum along the last axis (np.argmax: a NaN counts as the maximum) ----------------------
__global__ void __launch_bounds__(256) first_argmax_kernel(const double* __restrict__ value, int n, int A, int32_t* __restrict__ out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    double best = value[(size_t)b * A];
    int idx = 0;
    bool isn = best != best;
    for (int a = 1; a < A && !isn; a++) {
        const double v = value[(size_t)b * A + a];
        if (v != v) { idx = a; isn = true; }
        else if (v > best) { best = v; idx = a; }
    }
    out[b] = idx;
}

// ---- out[i][s] = alpha_a entry of tuple i; vsel_i = vsel + i*vselStride + (perAction ? action_i*O : 0) ---------------
__global__ void __launch_bounds__(256) assemble_kernel(const double* __restrict__ alphas, const int32_t* __restrict__ actions,
                                                       const int32_t* __restrict__ vsel, size_t vselStride, int perAction,
                                                       const int32_t* __restrict__ reachK, const double* __restrict__ rtoK,
                                                       const double* __restrict__ rbarT, double gamma, int S, int R, int O,
                                                       double* __restrict__ out, unsigned long long* __restrict__ hacc,
                                                       const int* __restrict__ nonfinite, int A, int nV) {
    extern __shared__ int s_vsel[];
    __shared__ unsigned long long sh[2][8];
    const int i = blockIdx.y, a = min(max(actions[i], 0), A - 1);       // indices are clamped: a bad tuple never reads out of bounds
    const int32_t* vs = vsel + (size_t)i * vselStride + (perAction ? (size_t)a * O : 0);
    for (int o = threadIdx.x; o < O; o += 256) s_vsel[o] = min(max(vs[o], 0), nV - 1);
    __syncthreads();
    const int s = blockIdx.x * 256 + threadIdx.x;
    unsigned long long h0 = 0, h1 = 0;
    if (s < S) {
        const double v = alpha_a_entry(alphas, S, R, O, s_vsel, reachK + (size_t)a * S * R, rtoK + (size_t)a * O * S * R,
                                       rbarT + (size_t)a * S, gamma, s, !*nonfinite);
        out[(size_t)i * S + s] = v;
        if (hacc) {
            const uint64_t w = (uint64_t)__double_as_longlong(v);
            const uint4 k = row_key_words(s);
            h0 = row_hash_term0(w, k);
            h1 = row_hash_term1(w, k);
        }
    }
    if (!hacc) return;
    // the row's 128-bit key, accumulated while the row is still in registers (same value as row_hash_kernel over the finished row)
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        h0 += __shfl_down_sync(0xffffffffu, h0, off);
        h1 += __shfl_down_sync(0xffffffffu, h1, off);
    }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = h0; sh[1][threadIdx.x >> 5] = h1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long x = 0, y = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) { x += sh[0][w]; y += sh[1][w]; }
        atomicAdd(&hacc[(size_t)i * 2], x);
        atomicAdd(&hacc[(size_t)i * 2 + 1], y);
    }
}

// ---- one evaluation sweep of a finite-state controller: out[i][s] = alpha_a entry of the tuple (actions[i], succ[i][.]) against the
//      n rows `in` (the assemble kernel's arithmetic, so out is bitwise what pbvi_backup_assemble gives for the same tuples).  Block per
//      (node i, 256 states), 1-D grid.  With stats != nullptr every block leaves {max d, -min d, max |d|} of d = out - in (rows paired by
//      index; NaN wins) in part[block]; the last block to finish reduces the parts into stats[3].
constexpr int CTRL_THREADS = 256;

__device__ __forceinline__ void ctrl_reduce3(double& a, double& b, double& c, bool& nan, double (*sh)[CTRL_THREADS / 32], int* shn) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        a = fmax(a, __shfl_down_sync(0xffffffffu, a, off));
        b = fmax(b, __shfl_down_sync(0xffffffffu, b, off));
        c = fmax(c, __shfl_down_sync(0xffffffffu, c, off));
    }
    const unsigned anyNan = __ballot_sync(0xffffffffu, nan);
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = a; sh[1][threadIdx.x >> 5] = b; sh[2][threadIdx.x >> 5] = c; shn[threadIdx.x >> 5] = anyNan != 0; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < CTRL_THREADS / 32; w++) {
            a = fmax(a, sh[0][w]);
            b = fmax(b, sh[1][w]);
            c = fmax(c, sh[2][w]);
            nan |= shn[w] != 0;
        }
        nan |= shn[0] != 0;
    }
}

__global__ void __launch_bounds__(CTRL_THREADS) controller_sweep_kernel(const double* __restrict__ in, int n, const int32_t* __restrict__ actions,
                                                                        const int32_t* __restrict__ succ, const int32_t* __restrict__ reachK,
                                                                        const double* __restrict__ rtoK, const double* __restrict__ rbarT,
                                                                        double gamma, int S, int R, int O, int A, int sBlocks, bool skipZero,
                                                                        double* __restrict__ out, double* __restrict__ part,
                                                                        unsigned int* __restrict__ done, double* __restrict__ stats) {
    extern __shared__ int s_vsel[];
    __shared__ double sh[3][CTRL_THREADS / 32];
    __shared__ int shn[CTRL_THREADS / 32];
    __shared__ bool s_last;
    const int i = blockIdx.x / sBlocks, s = (blockIdx.x % sBlocks) * CTRL_THREADS + threadIdx.x;
    const int a = min(max(actions[i], 0), A - 1);                      // indices are clamped: a bad node never reads out of bounds
    for (int o = threadIdx.x; o < O; o += CTRL_THREADS) s_vsel[o] = min(max(succ[(size_t)i * O + o], 0), n - 1);
    __syncthreads();
    double up = -INFINITY, down = -INFINITY, amax = 0.0;
    bool nan = false;
    if (s < S) {
        const double v = alpha_a_entry(in, S, R, O, s_vsel, reachK + (size_t)a * S * R, rtoK + (size_t)a * O * S * R, rbarT + (size_t)a * S,
                                       gamma, s, skipZero);
        out[(size_t)i * S + s] = v;
        if (stats) {
            const double d = __dadd_rn(v, -in[(size_t)i * S + s]);
            nan = d != d;
            up = d;
            down = -d;
            amax = fabs(d);
        }
    }
    if (!stats) return;
    ctrl_reduce3(up, down, amax, nan, sh, shn);
    if (threadIdx.x == 0) {
        const size_t b = blockIdx.x;
        part[3 * b] = nan ? NAN : up;
        part[3 * b + 1] = nan ? NAN : down;
        part[3 * b + 2] = nan ? NAN : amax;
        __threadfence();
        s_last = atomicAdd(done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const volatile double* pv = part;                                  // written by other blocks: bypass L1
    up = down = -INFINITY;
    amax = 0.0;
    nan = false;
    for (unsigned b = threadIdx.x; b < gridDim.x; b += CTRL_THREADS) {
        const double x = pv[3 * (size_t)b], y = pv[3 * (size_t)b + 1], z = pv[3 * (size_t)b + 2];
        nan |= x != x;
        up = fmax(up, x);
        down = fmax(down, y);
        amax = fmax(amax, z);
    }
    __syncthreads();                                                   // sh / shn are reused
    ctrl_reduce3(up, down, amax, nan, sh, shn);
    if (threadIdx.x == 0) {
        stats[0] = nan ? NAN : up;
        stats[1] = nan ? NAN : down;
        stats[2] = nan ? NAN : amax;
    }
}

// ---- up to maxSweeps evaluation sweeps in one cooperative launch (pbvi_controller_evaluate).  Blocks stride over the (node, 256-state)
//      items of controller_sweep_kernel with the same arithmetic; sweep k reads in0 (k = 0) or the rows sweep k-1 wrote, and writes
//      bufA (k even) or bufB (k odd).  Each block leaves max |d| of its items (NaN wins) in part[k & 1][block]; after the one grid
//      barrier of the sweep every block reduces all partials itself and so reaches the same stop decision (change < tol or NaN, or the
//      last sweep).  The two parities keep a block that has already entered sweep k+1 from overwriting slots of sweep k that a slower
//      block is still reading: slots of parity k & 1 are written again only after the barrier of sweep k+1, which every block passes
//      only after its reads.  A maximum is exact in any order, so the change values are bitwise those of pbvi_controller_sweep's stats.
//      When the last sweep wrote bufB, the blocks copy it into bufA (its writes are visible after the barrier).
__device__ __forceinline__ double ctrl_reduce_max(double v, bool nan, double* sh, int* shn) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, off));
    const unsigned anyNan = __ballot_sync(0xffffffffu, nan);
    __syncthreads();                                                   // sh / shn of the previous use have been read
    if ((threadIdx.x & 31) == 0) { sh[threadIdx.x >> 5] = v; shn[threadIdx.x >> 5] = anyNan != 0; }
    __syncthreads();
    bool n = false;
#pragma unroll
    for (int w = 0; w < CTRL_THREADS / 32; w++) {
        v = fmax(v, sh[w]);
        n |= shn[w] != 0;
    }
    return n ? NAN : v;
}

__global__ void __launch_bounds__(CTRL_THREADS) controller_evaluate_kernel(const double* __restrict__ in0, int n, const int32_t* __restrict__ actions,
                                                                           const int32_t* __restrict__ succ, const int32_t* __restrict__ reachK,
                                                                           const double* __restrict__ rtoK, const double* __restrict__ rbarT,
                                                                           double gamma, int S, int R, int O, int A, int sBlocks, bool skipZero,
                                                                           double tol, int maxSweeps, double* bufA, double* bufB, double* part,
                                                                           double* __restrict__ changes, int* __restrict__ sweepsOut) {
    extern __shared__ int s_vsel[];
    __shared__ double sh[CTRL_THREADS / 32];
    __shared__ int shn[CTRL_THREADS / 32];
    cg::grid_group grid = cg::this_grid();
    const int items = n * sBlocks;
    int k = 0;
    for (;; k++) {
        // rows written earlier in this launch are read with ld.global.cg, never through the read-only data cache
        const double* src = (k == 0) ? in0 : ((k & 1) ? bufA : bufB);
        double* dst = (k & 1) ? bufB : bufA;
        double amax = 0.0;
        bool nan = false;
        for (int it = blockIdx.x; it < items; it += gridDim.x) {
            const int i = it / sBlocks, s = (it % sBlocks) * CTRL_THREADS + threadIdx.x;
            const int a = min(max(actions[i], 0), A - 1);
            __syncthreads();                                           // s_vsel of the previous item has been used
            for (int o = threadIdx.x; o < O; o += CTRL_THREADS) s_vsel[o] = min(max(succ[(size_t)i * O + o], 0), n - 1);
            __syncthreads();
            if (s < S) {
                const double v = alpha_a_entry<true>(src, S, R, O, s_vsel, reachK + (size_t)a * S * R, rtoK + (size_t)a * O * S * R,
                                                     rbarT + (size_t)a * S, gamma, s, skipZero);
                dst[(size_t)i * S + s] = v;
                const double d = __dadd_rn(v, -__ldcg(src + (size_t)i * S + s));
                nan |= d != d;
                amax = fmax(amax, fabs(d));
            }
        }
        const double mine = ctrl_reduce_max(amax, nan, sh, shn);
        double* slots = part + (size_t)(k & 1) * gridDim.x;
        if (threadIdx.x == 0) slots[blockIdx.x] = mine;
        grid.sync();
        amax = 0.0;
        nan = false;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += CTRL_THREADS) {
            const double x = __ldcg(slots + b);
            nan |= x != x;
            amax = fmax(amax, x);
        }
        const double change = ctrl_reduce_max(amax, nan, sh, shn);
        if (changes && blockIdx.x == 0 && threadIdx.x == 0) changes[k] = change;
        if (!(change >= tol) || k + 1 == maxSweeps) break;           // converged, NaN, or out of sweeps: the same decision in every block
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *sweepsOut = k + 1;
    if (k & 1) {
        const size_t total = (size_t)n * S;
        for (size_t e = (size_t)blockIdx.x * CTRL_THREADS + threadIdx.x; e < total; e += (size_t)gridDim.x * CTRL_THREADS) bufA[e] = __ldcg(bufB + e);
    }
}

// ---- order[] = tuple indices grouped by action, every group padded with -1 to a multiple of G (so that a block of the grouped
//      assemble kernel sees one action only); counting sort in one block, the order inside an action is irrelevant.
//      order has room for n + A * (G - 1) entries and is pre-filled with -1.
__global__ void __launch_bounds__(256) action_order_kernel(const int32_t* __restrict__ actions, int n, int A, int G, int32_t* __restrict__ order) {
    extern __shared__ int s_cnt[];     // [A] counts, then running bases
    for (int a = threadIdx.x; a < A; a += 256) s_cnt[a] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += 256) atomicAdd(&s_cnt[min(max(actions[i], 0), A - 1)], 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int a = 0; a < A; a++) { const int c = s_cnt[a]; s_cnt[a] = run; run += (c + G - 1) / G * G; }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += 256) order[atomicAdd(&s_cnt[min(max(actions[i], 0), A - 1)], 1)] = i;
}

// ---- assemble for reachable_state_count == 1 and O <= OM: a block writes the same SPT*256-state slice of G tuples of ONE
//      action, so reach / RTO / Rbar of the slice are read once per block instead of once per tuple; what is left per element
//      is the O gathered alpha values, the two hash terms and the store.  The gathers of tuple g+1 are issued before the
//      arithmetic of tuple g (the loop is otherwise one exposed memory latency per tuple).  A thread owns SPT states (256 apart:
//      coalesced), which amortises the per-tuple reduction of the 128-bit key; the warp partials of all G tuples meet in shared
//      memory once, at the end.  Same arithmetic as alpha_a_entry (bit-identical rows).
template <int G, int OM, int SPT>
__global__ void __launch_bounds__(256) assemble_grouped_kernel(const double* __restrict__ alphas, const int32_t* __restrict__ actions,
                                                               const int32_t* __restrict__ vsel, const int32_t* __restrict__ order,
                                                               const int32_t* __restrict__ reachK, const double* __restrict__ rtoK,
                                                               const double* __restrict__ rbarT, double gamma, int S, int O,
                                                               double* __restrict__ out, unsigned long long* __restrict__ hacc,
                                                               const uint4* __restrict__ hashKeys, const int* __restrict__ nonfinite,
                                                               int A, int nV) {
    __shared__ int s_idx[G], s_v[G][OM];
    __shared__ unsigned long long sh[G][8][2];
    const int slot0 = blockIdx.y * G;
    if (threadIdx.x < G) s_idx[threadIdx.x] = order[slot0 + threadIdx.x];
    __syncthreads();
    if (s_idx[0] < 0) return;                        // padding block (uniform)
    if (threadIdx.x < G * OM) {
        const int g = threadIdx.x / OM, o = threadIdx.x % OM;
        s_v[g][o] = (s_idx[g] >= 0 && o < O) ? min(max(vsel[(size_t)s_idx[g] * O + o], 0), nV - 1) : 0;
    }
    const int a = min(max(actions[s_idx[0]], 0), A - 1);
    __syncthreads();
    const int sBase = blockIdx.x * (SPT * 256) + threadIdx.x;
    const bool skipZero = !*nonfinite;              // finite alphas: a zero RTO factor makes the term +-0.0 (see alpha_a_entry)
    bool need[SPT][OM], live[SPT];
    int landing[SPT];
    double rb[SPT], rto[SPT][OM];
    uint4 hk[SPT];
#pragma unroll
    for (int j = 0; j < SPT; j++) {
        const int s = sBase + j * 256;
        live[j] = s < S;
        landing[j] = live[j] ? reachK[(size_t)a * S + s] : 0;
        rb[j] = live[j] ? rbarT[(size_t)a * S + s] : 0.0;
        hk[j] = (hacc && live[j]) ? hashKeys[s] : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int o = 0; o < OM; o++) rto[j][o] = (live[j] && o < O) ? rtoK[((size_t)a * O + o) * S + s] : 0.0;
    }
#pragma unroll
    for (int j = 0; j < SPT; j++) {
        const bool skip = skipZero && !(rb[j] == 0.0 && signbit(rb[j]));
#pragma unroll
        for (int o = 0; o < OM; o++) need[j][o] = live[j] && o < O && !(skip && rto[j][o] == 0.0);
    }
    auto gather = [&](int g, double (&av)[SPT][OM]) {
#pragma unroll
        for (int j = 0; j < SPT; j++)
#pragma unroll
            for (int o = 0; o < OM; o++) av[j][o] = need[j][o] ? alphas[(size_t)s_v[g][o] * S + landing[j]] : 0.0;
    };
    auto finish = [&](int g, const double (&av)[SPT][OM]) {
        const int idx = s_idx[g];
        unsigned long long h0 = 0, h1 = 0;
#pragma unroll
        for (int j = 0; j < SPT; j++) {
            if (live[j]) {
                double tot = 0.0;
#pragma unroll
                for (int o = 0; o < OM; o++)
                    if (o < O) {
                        const double term = need[j][o] ? __dmul_rn(gamma, __dmul_rn(rto[j][o], av[j][o])) : 0.0;
                        tot = (o == 0) ? term : __dadd_rn(tot, term);
                    }
                const double v = __dadd_rn(rb[j], tot);
                out[(size_t)idx * S + sBase + j * 256] = v;
                if (hacc) {
                    const uint64_t w = (uint64_t)__double_as_longlong(v);
                    h0 += row_hash_term0(w, hk[j]);
                    h1 += row_hash_term1(w, hk[j]);
                }
            }
        }
        if (hacc) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                h0 += __shfl_down_sync(0xffffffffu, h0, off);
                h1 += __shfl_down_sync(0xffffffffu, h1, off);
            }
            if ((threadIdx.x & 31) == 0) { sh[g][threadIdx.x >> 5][0] = h0; sh[g][threadIdx.x >> 5][1] = h1; }
        }
    };
    static_assert(G % 2 == 0, "the tuple loop is unrolled in pairs (two gather buffers)");
    double avA[SPT][OM], avB[SPT][OM];
    gather(0, avA);
#pragma unroll
    for (int g = 0; g < G; g += 2) {
        const bool has1 = s_idx[g + 1] >= 0;                               // uniform over the block
        if (has1) gather(g + 1, avB);
        finish(g, avA);
        if (!has1) break;
        const bool has2 = g + 2 < G && s_idx[g + 2 < G ? g + 2 : 0] >= 0;
        if (has2) gather(g + 2, avA);
        finish(g + 1, avB);
        if (!has2) break;
    }
    if (!hacc) return;
    __syncthreads();
    if (threadIdx.x < G * 2) {
        const int g = threadIdx.x >> 1, which = threadIdx.x & 1;
        const int idx = s_idx[g];
        if (idx >= 0) {
            unsigned long long x = 0;
#pragma unroll
            for (int w = 0; w < 8; w++) x += sh[g][w][which];
            atomicAdd(&hacc[(size_t)idx * 2 + which], x);
        }
    }
}

template <int G, int OM, int SPT>
static void launch_assemble_grouped(pbvi_model* m, const double* d_alphas, int nV, const int32_t* d_actions, const int32_t* d_vsel,
                                    const int32_t* order, int nPad, double gamma, double* d_out, unsigned long long* hacc, const int* nonfinite,
                                    cudaStream_t st) {
    assemble_grouped_kernel<G, OM, SPT><<<dim3(ceil_div(m->S, SPT * 256), nPad / G), 256, 0, st>>>(
        d_alphas, d_actions, d_vsel, order, m->reachK, m->rtoK, m->rbarT, gamma, m->S, m->O, d_out, hacc, m->hashKeys, nonfinite, m->A, nV);
}

// =====================================================================================================================
// Small-model path (tiger, 4x4 grids: BASELINE configs[0] / [1]).  The general pipeline above is ~20 launches and four host
// synchronisations whatever the problem size -- 0.3 ms for a backup whose arithmetic takes microseconds.  Here ONE kernel does the whole
// per-belief part, one block per belief, everything in shared memory:
//   1. btilde[z][s'] = sum_{k: reach[a][k] = s'} RTO[a][o][k] * b[k / R]      (the un-normalised Belief.update, CSR over landing states)
//   2. v*[z] = first argmax_v btilde[z] . alpha_v                             (warp per z, np.argmax semantics incl. NaN)
//   3. value[a] = sum_s b[s] * alpha_a[s],  a* = first argmax_a               (alpha_a_entry: the reference's operation order)
//   4. row = alpha_{a*}, its 128-bit key, a*
// and pbvi_backup_small finishes the backup on the host side of the same call: rows, keys and actions come back in one copy, the
// ValueFunction constructor's dict semantics (first position, last action; keys confirmed with memcmp) run on at most a few
// thousand rows, and a gather kernel writes the surviving rows.  One synchronisation per backup.
constexpr int SMALL_THREADS = 128;

__global__ void __launch_bounds__(SMALL_THREADS) small_backup_kernel(const double* __restrict__ beliefs, const double* __restrict__ alphas,
                                                                     const int32_t* __restrict__ reachK, const double* __restrict__ rtoK,
                                                                     const double* __restrict__ rbarT, const int32_t* __restrict__ predPtr,
                                                                     const int32_t* __restrict__ predK, double gamma, int S, int R, int A, int O,
                                                                     int nV, double* __restrict__ rows, unsigned long long* __restrict__ keys,
                                                                     int32_t* __restrict__ actions) {
    extern __shared__ __align__(16) unsigned char small_smem[];
    const int nZ = A * O, K = S * R;
    double* sb = reinterpret_cast<double*>(small_smem);            // [S]
    double* sbt = sb + S;                                          // [nZ][S]
    double* sval = sbt + (size_t)nZ * S;                           // [A]
    int* svs = reinterpret_cast<int*>(sval + A);                   // [nZ]
    __shared__ unsigned long long sh[2][SMALL_THREADS / 32];
    __shared__ int s_bad, s_astar;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, b = blockIdx.x;
    const double* brow = beliefs + (size_t)b * S;
    if (tid == 0) s_bad = 0;
    __syncthreads();
    for (int s = tid; s < S; s += SMALL_THREADS) {
        const double v = brow[s];
        sb[s] = v;
        if (!(fabs(v) <= 1.79769313486231570e308)) s_bad = 1;      // NaN / inf belief entry: every score is NaN in the reference
    }
    __syncthreads();
    // 1. projections (bincount order, like belief_project_kernel)
    for (int i = tid; i < nZ * S; i += SMALL_THREADS) {
        const int z = i / S, sp = i - z * S, a = z / O;
        const int32_t* ptr = predPtr + (size_t)a * (S + 1);
        const int32_t* pk = predK + (size_t)a * K;
        const double* rto = rtoK + (size_t)z * K;
        double acc = 0.0;
        for (int j = ptr[sp]; j < ptr[sp + 1]; j++) {
            const int k = pk[j];
            acc = __dadd_rn(acc, __dmul_rn(rto[k], sb[R == 1 ? k : k / R]));
        }
        sbt[i] = acc;
    }
    __syncthreads();
    // 2. v*[z]: warp per z, lanes over v (ascending per lane), warp argmax with the lower index winning ties
    const bool bad = s_bad != 0;
    for (int z = warp; z < nZ; z += SMALL_THREADS / 32) {
        const double* bt = sbt + (size_t)z * S;
        double best = -INFINITY;
        int bidx = ARG_NONE;
        for (int v = lane; v < nV; v += 32) {
            const double* al = alphas + (size_t)v * S;
            double acc = 0.0;
            for (int s = 0; s < S; s++) acc = fma(bt[s], al[s], acc);
            argmax_append(best, bidx, acc, v);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, off);
            const int oi = __shfl_xor_sync(0xffffffffu, bidx, off);
            argmax_combine(best, bidx, ov, oi);
        }
        if (lane == 0) svs[z] = bad ? 0 : min(max(bidx, 0), nV - 1);
    }
    __syncthreads();
    // 3. value[a] and a*
    for (int a = warp; a < A; a += SMALL_THREADS / 32) {
        double part = 0.0;
        for (int s = lane; s < S; s += 32)
            part = fma(sb[s], alpha_a_entry(alphas, S, R, O, svs + a * O, reachK + (size_t)a * K, rtoK + (size_t)a * O * K, rbarT + (size_t)a * S,
                                            gamma, s, false), part);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
        if (lane == 0) sval[a] = part;
    }
    __syncthreads();
    if (tid == 0) {
        double best = sval[0];
        int idx = 0;
        for (int a = 1; a < A && best == best; a++) {
            const double v = sval[a];
            if (v != v || v > best) { best = v; idx = a; }
        }
        s_astar = idx;
        actions[b] = idx;
    }
    __syncthreads();
    // 4. the row of a* and its key
    const int a = s_astar;
    unsigned long long h0 = 0, h1 = 0;
    for (int s = tid; s < S; s += SMALL_THREADS) {
        const double v = alpha_a_entry(alphas, S, R, O, svs + a * O, reachK + (size_t)a * K, rtoK + (size_t)a * O * K, rbarT + (size_t)a * S, gamma,
                                       s, false);
        rows[(size_t)b * S + s] = v;
        const uint64_t w = (uint64_t)__double_as_longlong(v);
        const uint4 k = row_key_words(s);
        h0 += row_hash_term0(w, k);
        h1 += row_hash_term1(w, k);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        h0 += __shfl_down_sync(0xffffffffu, h0, off);
        h1 += __shfl_down_sync(0xffffffffu, h1, off);
    }
    if (lane == 0) { sh[0][warp] = h0; sh[1][warp] = h1; }
    __syncthreads();
    if (tid == 0) {
        unsigned long long x = 0, y = 0;
        for (int w = 0; w < SMALL_THREADS / 32; w++) { x += sh[0][w]; y += sh[1][w]; }
        keys[(size_t)b * 2] = row_hash_final0(x, S);
        keys[(size_t)b * 2 + 1] = row_hash_final1(y, S);
    }
}

__global__ void __launch_bounds__(128) gather_rows_kernel(const double* __restrict__ src, const int32_t* __restrict__ idx, int S,
                                                          double* __restrict__ dst) {
    const double* r = src + (size_t)idx[blockIdx.x] * S;
    for (int s = threadIdx.x; s < S; s += 128) dst[(size_t)blockIdx.x * S + s] = r[s];
}

__global__ void __launch_bounds__(256) hash_finalise_kernel(unsigned long long* __restrict__ h, int n, int rowLen) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    h[(size_t)i * 2] = row_hash_final0(h[(size_t)i * 2], rowLen);
    h[(size_t)i * 2 + 1] = row_hash_final1(h[(size_t)i * 2 + 1], rowLen);
}

// =====================================================================================================================
// Function attributes are per device: called by pbvi_model_create for the handle's device (current when called).
// ---- pbvi_backup_host_unique: the tuple (a*, v*[a*, :]) of every belief as a group key, and the tuples / actions of the chosen groups
__global__ void __launch_bounds__(256) tuple_keys_kernel(const int32_t* __restrict__ vstar, const int32_t* __restrict__ astar, int n, int A,
                                                         int O, uint32_t* __restrict__ keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int a = min(max(astar[i], 0), A - 1);
    keys[(size_t)i * (1 + O)] = (uint32_t)a;
    for (int o = 0; o < O; o++) keys[(size_t)i * (1 + O) + 1 + o] = (uint32_t)vstar[((size_t)i * A + a) * O + o];
}

__global__ void __launch_bounds__(256) tuple_take_kernel(const uint32_t* __restrict__ keys, const int32_t* __restrict__ first,
                                                         const int32_t* __restrict__ last, int u, int O, int32_t* __restrict__ actions,
                                                         int32_t* __restrict__ vsel, int32_t* __restrict__ rank) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= u) return;
    const uint32_t* k = keys + (size_t)first[g] * (1 + O);
    actions[g] = (int32_t)k[0];
    for (int o = 0; o < O; o++) vsel[(size_t)g * O + o] = (int32_t)k[1 + o];
    rank[g] = last[g];
}

__global__ void __launch_bounds__(256) take_int_kernel(const int32_t* __restrict__ src, const int32_t* __restrict__ idx, int n,
                                                       int32_t* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[idx[i]];
}

int configure_backup_kernels() {
    PBVI_CUDA(cudaFuncSetAttribute(score_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCORE_SMEM));
    PBVI_CUDA(cudaFuncSetAttribute(score_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCORE_SMEM));
    return PBVI_OK;
}

static int launch_score(pbvi_model* m, bool gather, ScoreParams& p, int nNt, int nMt, int nZ, cudaStream_t st) {
    // persistent: one block per SM pulls (z, belief tile, alpha tile) tiles from a queue
    PBVI_REQUIRE((long long)nNt * nMt * nZ < (1ll << 31), "too many score tiles");
    p.nMt = nMt; p.nNt = nNt; p.nzLaunch = nZ;
    p.tileCounter = m->d_signs + 4;
    PBVI_CUDA(cudaMemsetAsync(p.tileCounter, 0, sizeof(int), st));
    const int grid = std::min(m->sm_count, nNt * nMt * nZ);
    if (gather) score_kernel<true><<<grid, SCORE_THREADS_TOTAL, SCORE_SMEM, st>>>(p);
    else score_kernel<false><<<grid, SCORE_THREADS_TOTAL, SCORE_SMEM, st>>>(p);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

// beliefs x (alphaT or Gamma) with fused argmax.  nZ == 0: plain max_v b.alpha_v (one z, no RTO mask).
// outVal/outIdx [nB][max(nZ,1)].
static int score_argmax(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, bool backup,
                        double* outVal, int32_t* outIdx, cudaStream_t st) {
    const int S = m->S, R = m->R, nC = m->nChunks;
    const int nZ = backup ? m->nZ : 1;
    const int Vp = ceil_div(nV, BN) * BN, nNt = Vp / BN, nMt = ceil_div(nB, BM);
    PBVI_REQUIRE(nMt <= 65535, "too many beliefs in one call (limit 65535 * 64)");
    PBVI_REQUIRE(nZ <= 65535, "too many (action, observation) pairs");

    // S + 1 rows: row S is all zero.  The pad states of the last pipeline stage (S is rounded up to whole stages) gather THAT row, so
    // their contribution is 0 * 0 whatever the alphas hold (a pad that re-read a real row would turn an infinite alpha into NaN).
    PBVI_TAKE(alphaT, double, (size_t)(S + 1) * Vp);
    PBVI_TRY(transpose_alphas(m, d_alphas, nV, Vp, alphaT, st));
    PBVI_CUDA(cudaMemsetAsync(alphaT + (size_t)S * Vp, 0, (size_t)Vp * sizeof(double), st));

    PBVI_TAKE(bits, uint8_t, (size_t)nMt * nC);
    m->last_bits = bits;           // read again by the value pass of the same call
    PBVI_TAKE(beliefsP, double, (size_t)nMt * nC * NRG * A_GROUP_DOUBLES);
    PBVI_TAKE(rowBad, uint8_t, (size_t)nMt * BM);
    PBVI_CUDA(cudaMemsetAsync(m->d_signs, 0, 8 * sizeof(int), st));
    PBVI_CUDA(cudaMemsetAsync(rowBad, 0, (size_t)nMt * BM, st));
    // alpha-side occupancy first: its scan also decides whether anything may be skipped at all (SIGN_DENSE: non-finite alphas).
    // Gather path: per action; plain max_v path: one group; Gamma path (R > 1): scanned for the sign / finiteness flags only (a
    // Gamma built from a non-negative model and non-negative alphas is non-negative), its B operand is not masked.
    uint8_t* bLive = nullptr;
    int nG = 1, zPerG = 1;
    PBVI_TAKE(rowLive, uint8_t, (size_t)nNt * S);
    alpha_row_mask_kernel<<<(unsigned)ceil_div_sz((size_t)S * nNt * 32, 256), 256, 0, st>>>(alphaT, S, Vp, nNt, rowLive, m->d_signs);
    m->last_launches++;
    if (!backup || R == 1) {
        nG = backup ? m->A : 1;
        zPerG = backup ? m->O : 1;
        bLive = m->arena.take<uint8_t>((size_t)nNt * nG * nC);
        if (!bLive) return PBVI_ERR_OOM;
        chunk_alpha_mask_kernel<<<(unsigned)ceil_div_sz((size_t)nNt * nG * nC, 256), 256, 0, st>>>(rowLive, backup ? m->reachP : nullptr, S,
                                                                                                  m->Sp, nC, nG, nNt, bLive, m->d_signs);
        m->last_launches++;
    }
    belief_mask_kernel<<<dim3(ceil_div(nC, MASK_CHUNKS), nMt), 256, 0, st>>>(d_beliefs, nB, S, nC, bits, beliefsP, m->d_signs, rowBad);
    m->last_launches++;
    PBVI_REQUIRE((size_t)nZ * nNt <= 2147483647u, "too many (z, alpha tile) pairs");
    PBVI_TAKE(lists, uint2, (size_t)nMt * nZ * nNt * (nC / SUB));
    PBVI_TAKE(counts, int32_t, (size_t)nMt * nZ * nNt);
    build_chunk_lists_kernel<<<dim3(nZ * nNt, nMt), 32, 0, st>>>(bits, backup ? m->zMask : nullptr, bLive, nG, zPerG, nC, nZ, nNt, lists,
                                                                 counts, m->d_signs);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());

    PBVI_TAKE(pval, double, (size_t)nNt * NCW * nB * nZ);
    PBVI_TAKE(pidx, int32_t, (size_t)nNt * NCW * nB * nZ);
    PBVI_CUDA(cudaMemsetAsync(m->d_stats, 0, sizeof(unsigned long long), st));
    m->last_exec_scale = 2.0 * RG * (BN / NCW) * KC;     // per visited (chunk, row group, column quarter)
    m->last_dense_flops = 2.0 * nB * (double)nV * nZ * S;

    if (m->profile) PBVI_CUDA(cudaEventRecord(m->evScore0, st));
    ScoreParams p{};
    p.beliefsP = beliefsP; p.lists = lists; p.listCount = counts; p.pval = pval; p.pidx = pidx; p.stats = m->d_stats;
    p.nB = nB; p.S = S; p.Sp = m->Sp; p.V = nV; p.Vp = Vp; p.nChunks = nC; p.nStages = nC / SUB; p.nZ = nZ; p.O = m->O;
    if (!backup) {
        p.bmat = alphaT; p.zStrideB = 0; p.zOrder = nullptr;
        PBVI_TRY(launch_score(m, false, p, nNt, nMt, 1, st));
    } else if (R == 1) {
        p.bmat = alphaT; p.zStrideB = 0; p.zOrder = m->zOrder; p.reachP = m->reachP; p.rtoP = m->rtoP;
        PBVI_TRY(launch_score(m, true, p, nNt, nMt, nZ, st));
    } else {
        // Gamma projection in groups of z bounded by ~8 GB of scratch
        const size_t perZ = (size_t)(S + 1) * Vp * sizeof(double);             // + the zero row of the pad states
        const int zGroup = (int)std::max<size_t>(1, std::min<size_t>(nZ, (size_t(8) << 30) / perZ));
        PBVI_TAKE(gammaT, double, (size_t)zGroup * (S + 1) * Vp);
        PBVI_CUDA(cudaMemset2DAsync(gammaT + (size_t)S * Vp, perZ, 0, (size_t)Vp * sizeof(double), (size_t)zGroup, st));
        for (int z0 = 0; z0 < nZ; z0 += zGroup) {
            const int nz = std::min(zGroup, nZ - z0);
            gamma_project_kernel<<<dim3(ceil_div(S, 8), nz), 256, 0, st>>>(alphaT, m->reachK, m->rtoK, m->zOrder, z0, S, R, m->O, Vp, gammaT,
                                                                           m->d_signs);
            m->last_launches++;
            p.bmat = gammaT; p.zStrideB = (size_t)(S + 1) * Vp; p.zOrder = m->zOrder + z0;
            PBVI_TRY(launch_score(m, false, p, nNt, nMt, nz, st));
        }
    }
    if (m->profile) { PBVI_CUDA(cudaEventRecord(m->evScore1, st)); m->score_timed = true; }
    const size_t n = (size_t)nB * nZ;
    combine_tiles_kernel<<<(unsigned)ceil_div_sz(n, 256), 256, 0, st>>>(pval, pidx, nNt * NCW, n, nZ, nV, rowBad, outVal, outIdx);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

static int check_backup_args(const pbvi_model* m, const void* beliefs, int nB, const void* alphas, int nV, double gamma) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(nB >= 0 && nV > 0, "need nB >= 0 beliefs and nV > 0 alpha vectors");
    PBVI_REQUIRE(nB == 0 || beliefs != nullptr, "beliefs pointer is NULL");
    PBVI_REQUIRE(alphas != nullptr, "alphas pointer is NULL");
    PBVI_REQUIRE(gamma > 0.0, "gamma must be positive (the score kernel drops it as an argmax-invariant scale)");
    return PBVI_OK;
}

static int select_impl(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double gamma,
                       int32_t* d_vstar, double* d_value, int32_t* d_astar, cudaStream_t st) {
    if (nB == 0) return PBVI_OK;
    double* maxscore = nullptr;
    if (d_value || d_astar) {
        maxscore = m->arena.take<double>((size_t)nB * m->nZ);
        if (!maxscore) return PBVI_ERR_OOM;
    }
    PBVI_TRY(score_argmax(m, d_beliefs, nB, d_alphas, nV, true, maxscore, d_vstar, st));
    if (!d_value && !d_astar) return PBVI_OK;
    const int needExact = d_value ? 1 : 0;        // values requested: every action that could win is summed in reference order
    if (!d_value) {
        d_value = m->arena.take<double>((size_t)nB * m->A);
        if (!d_value) return PBVI_ERR_OOM;
    }
    PBVI_REQUIRE(nB <= 65535 * BM, "too many beliefs in one call");
    PBVI_TAKE(approx, double, (size_t)nB * m->A);
    approx_value_kernel<<<(unsigned)ceil_div_sz((size_t)nB * m->A * 32, 256), 256, 0, st>>>(d_beliefs, maxscore, m->rbarNzPtr, m->rbarNzIdx,
                                                                                          m->rbarNzVal, gamma, m->S, m->A, m->O, nB, approx);
    m->last_launches++;
    // grid.y is limited to 65535: walk the beliefs in slabs
    const double relMargin = std::max(1e-10, 4.0 * (double)m->S * m->R * m->O * 1.1102230246251565e-16);
    for (int b0 = 0; b0 < nB; b0 += 65535) {
        const int nb = std::min(65535, nB - b0);
        backup_value_kernel<<<dim3(m->A, nb), 256, m->O * sizeof(int), st>>>(
            d_beliefs, d_alphas, d_vstar, m->reachK, m->rtoK, m->rbarT, approx, m->d_signs, m->model_nonneg ? 1 : 0, m->last_bits, m->nChunks,
            b0, gamma, m->S, m->R, m->A, m->O, nV, needExact, relMargin, d_value);
        m->last_launches++;
    }
    if (d_astar) {
        first_argmax_kernel<<<ceil_div(nB, 256), 256, 0, st>>>(d_value, nB, m->A, d_astar);
        m->last_launches++;
    }
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

static int assemble_impl(pbvi_model* m, const double* d_alphas, int nV, double gamma, const int32_t* d_actions, const int32_t* d_vsel,
                         size_t vselStride, int perAction, int n, double* d_out, uint64_t* d_hash, cudaStream_t st) {
    unsigned long long* hacc = reinterpret_cast<unsigned long long*>(d_hash);
    if (hacc) PBVI_CUDA(cudaMemsetAsync(hacc, 0, (size_t)n * 2 * sizeof(unsigned long long), st));
    // zero-RTO terms are skipped only when every alpha (and gamma) is finite: one streaming pass over the alphas decides
    int* nonfinite = m->d_signs + 3;
    const int gammaBad = (fabs(gamma) <= 1.79769313486231570e308) ? 0 : 1;
    PBVI_CUDA(cudaMemsetAsync(nonfinite, gammaBad, sizeof(int), st));
    nonfinite_scan_kernel<<<m->sm_count * 8, 256, 0, st>>>(d_alphas, (size_t)nV * m->S, nonfinite);
    m->last_launches++;
#ifndef PBVI_ASM_G
#define PBVI_ASM_G 8
#endif
#ifndef PBVI_ASM_SPT
#define PBVI_ASM_SPT 2
#endif
    constexpr int G = PBVI_ASM_G, SPT = PBVI_ASM_SPT;      // tuples per block / states per thread of the grouped assemble kernel (A/B builds)
    if (m->R == 1 && m->O <= 4 && !perAction && n >= 4 * G && (size_t)m->A * sizeof(int) <= 48 * 1024 &&
        ((long long)n + (long long)m->A * (G - 1)) / G + 1 <= 65535) {            // grid.y of the grouped kernel
        const int nPad = ceil_div(n + m->A * (G - 1), G) * G;
        PBVI_TAKE(order, int32_t, (size_t)nPad);
        PBVI_CUDA(cudaMemsetAsync(order, 0xFF, (size_t)nPad * sizeof(int32_t), st));
        action_order_kernel<<<1, 256, m->A * sizeof(int), st>>>(d_actions, n, m->A, G, order);
        if (m->O <= 2) launch_assemble_grouped<G, 2, SPT>(m, d_alphas, nV, d_actions, d_vsel, order, nPad, gamma, d_out, hacc, nonfinite, st);
        else if (m->O == 3) launch_assemble_grouped<G, 3, SPT>(m, d_alphas, nV, d_actions, d_vsel, order, nPad, gamma, d_out, hacc, nonfinite, st);
        else launch_assemble_grouped<G, 4, SPT>(m, d_alphas, nV, d_actions, d_vsel, order, nPad, gamma, d_out, hacc, nonfinite, st);
        m->last_launches += 2;
        if (hacc) {
            hash_finalise_kernel<<<ceil_div(n, 256), 256, 0, st>>>(hacc, n, m->S);
            m->last_launches++;
        }
        PBVI_CUDA(cudaGetLastError());
        return PBVI_OK;
    }
    for (int i0 = 0; i0 < n; i0 += 65535) {
        const int ni = std::min(65535, n - i0);
        assemble_kernel<<<dim3(ceil_div(m->S, 256), ni), 256, m->O * sizeof(int), st>>>(
            d_alphas, d_actions + i0, d_vsel + (size_t)i0 * vselStride, vselStride, perAction, m->reachK, m->rtoK, m->rbarT, gamma,
            m->S, m->R, m->O, d_out + (size_t)i0 * m->S, hacc ? hacc + (size_t)i0 * 2 : nullptr, nonfinite, m->A, nV);
        m->last_launches++;
    }
    if (hacc) {
        hash_finalise_kernel<<<ceil_div(n, 256), 256, 0, st>>>(hacc, n, m->S);
        m->last_launches++;
    }
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

}  // namespace pbvi

using namespace pbvi;

extern "C" int pbvi_backup_select(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double gamma,
                                  int32_t* d_vstar, double* d_value, int32_t* d_astar, void* stream) {
    PBVI_TRY(check_backup_args(m, d_beliefs, nB, d_alphas, nV, gamma));
    PBVI_REQUIRE(nB == 0 || d_vstar != nullptr, "v_star output is required");
    PBVI_CUDA(cudaSetDevice(m->device));
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    m->last_launches = 0;
    return select_impl(m, d_beliefs, nB, d_alphas, nV, gamma, d_vstar, d_value, d_astar, (cudaStream_t)stream);
}

extern "C" int pbvi_backup_assemble(pbvi_model* m, const double* d_alphas, int nV, double gamma, const int32_t* d_actions,
                                    const int32_t* d_vsel, int n, double* d_out, uint64_t* d_hash, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n >= 0 && nV > 0, "need n >= 0 tuples and nV > 0 alpha vectors");
    if (n == 0) return PBVI_OK;
    PBVI_REQUIRE(d_alphas && d_actions && d_vsel && d_out, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    m->last_launches = 0;
    return assemble_impl(m, d_alphas, nV, gamma, d_actions, d_vsel, (size_t)m->O, 0, n, d_out, d_hash, (cudaStream_t)stream);
}

extern "C" int pbvi_controller_sweep(pbvi_model* m, const double* d_in, int n, double gamma, const int32_t* d_actions, const int32_t* d_succ,
                                     double* d_out, double* d_stats3, void* stream) {
    PBVI_REQUIRE(d_in && d_actions && d_succ && d_out, "NULL pointer argument");
    PBVI_REQUIRE(n >= 1, "need n >= 1 controller nodes");
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    const int sBlocks = ceil_div(m->S, CTRL_THREADS);
    PBVI_REQUIRE((long long)n * sBlocks <= 0x7fffffffLL, "too many controller nodes in one call");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, st));
    m->last_launches = 0;
    const unsigned nBlocks = (unsigned)((long long)n * sBlocks);
    double* part = nullptr;
    unsigned int* done = nullptr;
    if (d_stats3) {
        part = m->arena.take<double>((size_t)nBlocks * 3);
        done = m->arena.take<unsigned int>(1);
        if (!part || !done) return PBVI_ERR_OOM;
        PBVI_CUDA(cudaMemsetAsync(done, 0, sizeof(unsigned int), st));
    }
    // the rows are finite (the caller's contract), so zero-RTO terms are skipped exactly as pbvi_backup_assemble skips them for finite alphas
    const bool skipZero = fabs(gamma) <= 1.79769313486231570e308;
    controller_sweep_kernel<<<nBlocks, CTRL_THREADS, m->O * sizeof(int), st>>>(d_in, n, d_actions, d_succ, m->reachK, m->rtoK, m->rbarT, gamma,
                                                                               m->S, m->R, m->O, m->A, sBlocks, skipZero, d_out, part, done,
                                                                               d_stats3);
    m->last_launches++;
    PBVI_CUDA(cudaGetLastError());
    return PBVI_OK;
}

extern "C" int pbvi_controller_evaluate(pbvi_model* m, const double* d_in, int n, double gamma, const int32_t* d_actions, const int32_t* d_succ,
                                        double tol, int max_sweeps, double* d_out, double* d_changes, int* h_sweeps, void* stream) {
    PBVI_REQUIRE(d_in && d_actions && d_succ && d_out && h_sweeps, "NULL pointer argument");
    PBVI_REQUIRE(n >= 1, "need n >= 1 controller nodes");
    PBVI_REQUIRE(max_sweeps >= 1, "need max_sweeps >= 1");
    PBVI_REQUIRE(tol == tol, "tol must not be NaN");
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    const int sBlocks = ceil_div(m->S, CTRL_THREADS);
    PBVI_REQUIRE((long long)n * sBlocks <= 0x7fffffffLL, "too many controller nodes in one call");
    PBVI_REQUIRE(d_in != d_out, "d_in and d_out must be different buffers");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, st));
    m->last_launches = 0;
    const size_t smem = (size_t)m->O * sizeof(int);
    int perSM = 0;
    PBVI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, controller_evaluate_kernel, CTRL_THREADS, smem));
    if (perSM < 1) {
        set_error("pbvi_controller_evaluate: the kernel cannot be resident with %zu bytes of shared memory", smem);
        return PBVI_ERR_UNSUPPORTED;
    }
    // every block must be resident for the grid barrier; a grid larger than the work would only add blocks to each barrier
    const int nBlocks = (int)std::min<long long>((long long)perSM * m->sm_count, (long long)n * sBlocks);
    PBVI_TAKE(bufB, double, (size_t)n * m->S);
    PBVI_TAKE(part, double, (size_t)2 * nBlocks);
    PBVI_TAKE(d_sweeps, int, 1);
    const bool skipZero = fabs(gamma) <= 1.79769313486231570e308;   // as pbvi_controller_sweep
    int S = m->S, R = m->R, O = m->O, A = m->A;
    void* args[] = {(void*)&d_in, (void*)&n, (void*)&d_actions, (void*)&d_succ, (void*)&m->reachK, (void*)&m->rtoK, (void*)&m->rbarT,
                    (void*)&gamma, (void*)&S, (void*)&R, (void*)&O, (void*)&A, (void*)&sBlocks, (void*)&skipZero, (void*)&tol,
                    (void*)&max_sweeps, (void*)&d_out, (void*)&bufB, (void*)&part, (void*)&d_changes, (void*)&d_sweeps};
    PBVI_CUDA(cudaLaunchCooperativeKernel((const void*)controller_evaluate_kernel, dim3(nBlocks), dim3(CTRL_THREADS), args, smem, st));
    m->last_launches++;
    int sweeps = 0;
    PBVI_CUDA(cudaMemcpyAsync(&sweeps, d_sweeps, sizeof(int), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    *h_sweeps = sweeps;
    return PBVI_OK;
}

extern "C" int pbvi_backup(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double gamma,
                           double* d_out_alpha, int32_t* d_out_action, int32_t* d_out_vstar, double* d_out_value, void* stream) {
    PBVI_TRY(check_backup_args(m, d_beliefs, nB, d_alphas, nV, gamma));
    if (nB == 0) return PBVI_OK;
    PBVI_REQUIRE(d_out_alpha && d_out_action, "alpha / action outputs are required");
    PBVI_CUDA(cudaSetDevice(m->device));
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    m->last_launches = 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (!d_out_vstar) {
        d_out_vstar = m->arena.take<int32_t>((size_t)nB * m->nZ);
        if (!d_out_vstar) return PBVI_ERR_OOM;
    }
    PBVI_TRY(select_impl(m, d_beliefs, nB, d_alphas, nV, gamma, d_out_vstar, d_out_value, d_out_action, st));
    return assemble_impl(m, d_alphas, nV, gamma, d_out_action, d_out_vstar, (size_t)m->nZ, 1, nB, d_out_alpha, nullptr, st);
}

// Host buffers in, host buffers out, as a two-deep chunk pipeline: while the kernels of chunk k run on the caller's stream, the beliefs
// of chunk k + 1 arrive on an upload stream and the alpha rows of chunk k - 1 leave on a download stream (PCIe is full duplex; rows are
// independent given the alphas, so a chunk is a complete backup of its beliefs).  With pinned host buffers the three overlap -- on the
// bench workload (10 000 x 1 000, 1.76 GB each way) the call is bound by the link instead of by link + kernels + link; with pageable
// buffers the copies are staged by the driver and the call degrades to the sequential form, results unchanged.
constexpr int HOST_CHUNK_ROWS = 2048;

extern "C" int pbvi_backup_host(pbvi_model* m, const double* h_beliefs, int nB, const double* h_alphas, int nV, double gamma,
                                double* h_out_alpha, int32_t* h_out_action, void* stream) {
    PBVI_TRY(check_backup_args(m, h_beliefs, nB, h_alphas, nV, gamma));
    if (nB == 0) return PBVI_OK;
    PBVI_REQUIRE(h_out_alpha && h_out_action, "alpha / action outputs are required");
    PBVI_CUDA(cudaSetDevice(m->device));
    if (m->hostIn) {      // a previous host call that returned early (an error) may have left copies in flight on the side streams
        PBVI_CUDA(cudaStreamSynchronize(m->hostIn));
        PBVI_CUDA(cudaStreamSynchronize(m->hostOut));
    }
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    m->last_launches = 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (!m->hostIn) {
        PBVI_CUDA(cudaStreamCreateWithFlags(&m->hostIn, cudaStreamNonBlocking));
        PBVI_CUDA(cudaStreamCreateWithFlags(&m->hostOut, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            PBVI_CUDA(cudaEventCreateWithFlags(&m->evIn[i], cudaEventDisableTiming));
            PBVI_CUDA(cudaEventCreateWithFlags(&m->evDone[i], cudaEventDisableTiming));
            PBVI_CUDA(cudaEventCreateWithFlags(&m->evOut[i], cudaEventDisableTiming));
        }
    }
    const size_t S = m->S;
    const int rows = std::min(nB, HOST_CHUNK_ROWS);
    PBVI_TAKE(d_a, double, (size_t)nV * S);
    PBVI_TAKE(d_act, int32_t, (size_t)nB);
    double* d_b[2];
    double* d_out[2];
    for (int i = 0; i < 2; i++) {
        d_b[i] = m->arena.take<double>((size_t)rows * S);
        d_out[i] = m->arena.take<double>((size_t)rows * S);
        if (!d_b[i] || !d_out[i]) return PBVI_ERR_OOM;
    }
    PBVI_TAKE(d_vs, int32_t, (size_t)rows * m->nZ);
    // the staging buffers above are scratch of THIS call: the side streams may touch them only after everything the caller's stream
    // held before (an earlier call's kernels on the same arena) is done
    PBVI_CUDA(cudaEventRecord(m->evDone[0], st));
    PBVI_CUDA(cudaStreamWaitEvent(m->hostIn, m->evDone[0], 0));
    PBVI_CUDA(cudaStreamWaitEvent(m->hostOut, m->evDone[0], 0));
    PBVI_CUDA(cudaMemcpyAsync(d_a, h_alphas, (size_t)nV * S * sizeof(double), cudaMemcpyHostToDevice, st));
    const pbvi::Arena::Mark mark = m->arena.mark();
    int launches = 0;
    for (int lo = 0, k = 0; lo < nB; lo += rows, k++) {
        const int n = std::min(rows, nB - lo), b = k & 1;
        if (k >= 2) PBVI_CUDA(cudaStreamWaitEvent(m->hostIn, m->evDone[b], 0));        // chunk k - 2 has read d_b[b]
        PBVI_CUDA(cudaMemcpyAsync(d_b[b], h_beliefs + (size_t)lo * S, (size_t)n * S * sizeof(double), cudaMemcpyHostToDevice, m->hostIn));
        PBVI_CUDA(cudaEventRecord(m->evIn[b], m->hostIn));
        PBVI_CUDA(cudaStreamWaitEvent(st, m->evIn[b], 0));
        if (k >= 2) PBVI_CUDA(cudaStreamWaitEvent(st, m->evOut[b], 0));                // the rows of chunk k - 2 have left d_out[b]
        m->arena.rewind(mark);
        m->last_launches = 0;
        PBVI_TRY(select_impl(m, d_b[b], n, d_a, nV, gamma, d_vs, nullptr, d_act + lo, st));
        PBVI_TRY(assemble_impl(m, d_a, nV, gamma, d_act + lo, d_vs, (size_t)m->nZ, 1, n, d_out[b], nullptr, st));
        launches += m->last_launches;
        PBVI_CUDA(cudaEventRecord(m->evDone[b], st));
        PBVI_CUDA(cudaStreamWaitEvent(m->hostOut, m->evDone[b], 0));
        PBVI_CUDA(cudaMemcpyAsync(h_out_alpha + (size_t)lo * S, d_out[b], (size_t)n * S * sizeof(double), cudaMemcpyDeviceToHost, m->hostOut));
        PBVI_CUDA(cudaEventRecord(m->evOut[b], m->hostOut));
    }
    m->last_launches = launches;
    PBVI_CUDA(cudaMemcpyAsync(h_out_action, d_act, (size_t)nB * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    PBVI_CUDA(cudaStreamSynchronize(m->hostOut));
    PBVI_CUDA(cudaStreamSynchronize(m->hostIn));
    return PBVI_OK;
}

// ---- pageable host buffers (NumPy arrays) ------------------------------------------------------------------------------------------
// cudaMemcpyAsync from / to pageable memory is staged by the driver at a fraction of the link rate and blocks the calling thread, which
// the packed pipeline needs for shipping slabs.  Pageable alphas / output rows go through the handle's own pinned staging instead,
// moved by a few host threads (a core copies ~8 GB/s; the 176 MB of the bench's alphas take 3 ms on 15 threads).
static bool host_pointer_is_pinned(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}

static void* io_staging(pbvi_model* m, size_t bytes) {
    if (m->h_io_bytes < bytes) {
        if (m->h_io) cudaFreeHost(m->h_io);
        m->h_io = nullptr;
        m->h_io_bytes = 0;
        if (cudaHostAlloc(&m->h_io, bytes, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            m->h_io = nullptr;
            return nullptr;
        }
        m->h_io_bytes = bytes;
    }
    return m->h_io;
}

static void parallel_memcpy(void* dst, const void* src, size_t bytes) {
    const unsigned hw = std::thread::hardware_concurrency();
    const int T = (int)std::max<size_t>(1, std::min<size_t>({(size_t)(hw > 1 ? hw - 1 : 1), (size_t)32, bytes >> 22}));   // >= 4 MB per thread
    if (T == 1) { std::memcpy(dst, src, bytes); return; }
    std::vector<std::thread> th;
    const size_t slice = ((bytes / T) + 63) & ~size_t(63);
    for (int t = 0; t < T; t++) {
        const size_t lo = std::min(bytes, (size_t)t * slice), hi = std::min(bytes, lo + slice);
        if (hi <= lo) continue;
        bool spawned = false;
        try {                                                       // no C++ exception may cross the C ABI
            th.emplace_back([=] { std::memcpy(static_cast<char*>(dst) + lo, static_cast<const char*>(src) + lo, hi - lo); });
            spawned = true;
        } catch (...) {
        }
        if (!spawned) std::memcpy(static_cast<char*>(dst) + lo, static_cast<const char*>(src) + lo, hi - lo);
    }
    for (auto& x : th) x.join();
}

// ---- upload + select of a host-resident belief set, PACKED transport (the C form of PBVI_Solver._select_streamed) --------------------
// Sparse belief rows cross the link as [bitmap over 4-double chunks | the non-zero chunks]: host threads pack slabs of 64 rows into
// the handle's pinned staging (pbvi_pack_slabs_host), this thread ships every finished slab on the upload stream, pbvi_unpack_rows
// rebuilds the dense rows in HBM on a second stream and the select kernels follow chunk by chunk on the caller's stream.  The
// caller's belief buffer is only ever read by the host cores, so it may be pageable (a NumPy array) at no cost -- the dense pipeline
// needs page-locked rows to overlap anything.  *packed = false (nothing done): the rows are too dense (or too few) to be worth it.
constexpr int PACK_SLAB_ROWS = 64;
constexpr double PACK_MAX_DENSITY = 0.6;

static int host_select_packed(pbvi_model* m, const double* h_beliefs, int nB, const double* d_a, int nV, double gamma, int32_t* d_vs,
                              int32_t* d_act, cudaStream_t st, int* launches, bool* packed) {
    *packed = false;
    const int S = m->S, SL = PACK_SLAB_ROWS;
    const int nC = (S + 3) / 4, W = (nC + 31) / 32;
    if (nB < 2048) return PBVI_OK;
    {   // density of the first rows, at chunk granularity
        const int probe = std::min(nB, 8);
        long long live = 0;
        for (int i = 0; i < probe; i++)
            for (int c = 0; c < nC; c++) {
                bool nz = false;
                for (int j = 4 * c; j < std::min(S, 4 * c + 4) && !nz; j++) {
                    uint64_t w;
                    std::memcpy(&w, h_beliefs + (size_t)i * S + j, sizeof(w));
                    nz = w != 0;
                }
                live += nz ? 1 : 0;
            }
        if ((double)live > PACK_MAX_DENSITY * (double)probe * nC) return PBVI_OK;
    }
    const int n_slabs = ceil_div(nB, SL);
    const size_t region = (size_t)SL * nC * 4 + 4;                 // doubles per slab: worst case + the packer's one-chunk slack
    auto up256 = [](size_t b) { return (b + 255) & ~size_t(255); };
    const size_t bmBytes = up256((size_t)nB * W * 4), rsBytes = up256((size_t)n_slabs * (SL + 1) * 4), pkBytes = up256((size_t)n_slabs * region * 8),
                 totBytes = up256((size_t)n_slabs * 8);
    const size_t need = bmBytes + rsBytes + pkBytes + totBytes;
    if (m->h_pack_bytes < need) {
        if (m->h_pack) cudaFreeHost(m->h_pack);
        m->h_pack = nullptr;
        m->h_pack_bytes = 0;
        if (cudaHostAlloc(&m->h_pack, need, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            m->h_pack = nullptr;
            return PBVI_OK;                                      // no pinned memory for the staging: the dense pipeline does the job
        }
        m->h_pack_bytes = need;
    }
    char* hp = static_cast<char*>(m->h_pack);
    uint32_t* h_bm = reinterpret_cast<uint32_t*>(hp);
    int32_t* h_rs = reinterpret_cast<int32_t*>(hp + bmBytes);
    double* h_pk = reinterpret_cast<double*>(hp + bmBytes + rsBytes);
    int64_t* h_tot = reinterpret_cast<int64_t*>(hp + bmBytes + rsBytes + pkBytes);
    for (int i = 0; i < n_slabs; i++) h_tot[i] = -1;
    PBVI_TAKE(d_bm, uint32_t, (size_t)nB * W);
    PBVI_TAKE(d_rs, int32_t, (size_t)n_slabs * (SL + 1));
    PBVI_TAKE(d_pk, double, (size_t)n_slabs * region);
    PBVI_TAKE(d_full, double, (size_t)nB * S);
    // the staging above is scratch of this call: the side streams may touch it only after what the caller's stream held before
    PBVI_CUDA(cudaEventRecord(m->evDone[0], st));
    PBVI_CUDA(cudaStreamWaitEvent(m->hostIn, m->evDone[0], 0));
    PBVI_CUDA(cudaStreamWaitEvent(m->hostOut, m->evDone[0], 0));

    const unsigned hw = std::thread::hardware_concurrency();
    const int T = std::max(1, std::min({32, (int)(hw > 1 ? hw - 1 : 1), n_slabs}));     // one core stays with this thread
    std::vector<std::thread> packers;
    int started = 0;
    try {                                                           // no C++ exception may cross the C ABI
        packers.reserve(T);
        for (; started < T; started++) {
            const int t = started;
            packers.emplace_back([=] { pbvi_pack_slabs_host(h_beliefs, nB, S, SL, t, T, h_bm, h_rs, h_pk, (int64_t)region, h_tot); });
        }
    } catch (...) {
    }
    auto join_all = [&] { for (auto& th : packers) if (th.joinable()) th.join(); };
    for (int t = started; t < T; t++)                               // threads the system refused: their slabs are packed here, now
        pbvi_pack_slabs_host(h_beliefs, nB, S, SL, t, T, h_bm, h_rs, h_pk, (int64_t)region, h_tot);

    const int unit = SL * std::min(T, 16);                          // one round of the packers: ready after ONE slab time
    const pbvi::Arena::Mark mark = m->arena.mark();
    int rc = PBVI_OK, shipped = 0;                                  // slabs whose copies are enqueued
    int lo = 0, size = unit;
    while (lo < nB && rc == PBVI_OK) {
        int hi = std::min(nB, lo + size);
        if (nB - hi < unit) hi = nB;                                // a tail shorter than one unit joins the last chunk
        const int s1 = ceil_div(hi, SL);
        for (; shipped < s1 && rc == PBVI_OK; shipped++) {
            int64_t total;
            unsigned spins = 0;
            while ((total = __atomic_load_n(&h_tot[shipped], __ATOMIC_ACQUIRE)) == -1)
                if (++spins % 64 == 0) std::this_thread::yield();
            if (total < 0) { set_error("packing the host rows failed"); rc = PBVI_ERR_BAD_ARG; break; }
            if (total > 0 && cudaMemcpyAsync(d_pk + (size_t)shipped * region, h_pk + (size_t)shipped * region, (size_t)total * 32,
                                             cudaMemcpyHostToDevice, m->hostIn) != cudaSuccess) { set_error("cudaMemcpyAsync failed"); rc = PBVI_ERR_CUDA; }
        }
        if (rc != PBVI_OK) break;
        const int s0 = lo / SL;
        bool ok = cudaMemcpyAsync(d_bm + (size_t)lo * W, h_bm + (size_t)lo * W, (size_t)(hi - lo) * W * 4, cudaMemcpyHostToDevice, m->hostIn) == cudaSuccess;
        ok = ok && cudaMemcpyAsync(d_rs + (size_t)s0 * (SL + 1), h_rs + (size_t)s0 * (SL + 1), (size_t)(s1 - s0) * (SL + 1) * 4, cudaMemcpyHostToDevice,
                                   m->hostIn) == cudaSuccess;
        ok = ok && cudaEventRecord(m->evIn[0], m->hostIn) == cudaSuccess && cudaStreamWaitEvent(m->hostOut, m->evIn[0], 0) == cudaSuccess;
        if (!ok) { set_error("CUDA error while shipping packed rows: %s", cudaGetErrorString(cudaGetLastError())); rc = PBVI_ERR_CUDA; break; }
        m->last_launches = 0;
        rc = unpack_rows_launch(m, d_bm + (size_t)lo * W, d_rs + (size_t)s0 * (SL + 1), d_pk + (size_t)s0 * region, hi - lo, S, SL,
                                (long long)(region / 4), d_full + (size_t)lo * S, m->hostOut);
        if (rc != PBVI_OK) break;
        ok = cudaEventRecord(m->evOut[0], m->hostOut) == cudaSuccess && cudaStreamWaitEvent(st, m->evOut[0], 0) == cudaSuccess;
        if (!ok) { set_error("CUDA error: %s", cudaGetErrorString(cudaGetLastError())); rc = PBVI_ERR_CUDA; break; }
        m->arena.rewind(mark);
        rc = select_impl(m, d_full + (size_t)lo * S, hi - lo, d_a, nV, gamma, d_vs + (size_t)lo * m->nZ, nullptr, d_act + lo, st);
        *launches += m->last_launches;
        lo = hi;
        size = std::min(3 * unit, 2 * size);
    }
    join_all();
    m->arena.rewind(mark);
    if (rc == PBVI_OK) *packed = true;
    return rc;
}

// The reference's whole PBVI_Solver.backup (src/pomdp.py:1447-1524, belief_dominance_prune = False) from host buffers in one call:
// chunked upload behind the select kernels as in pbvi_backup_host, then -- what the reference does with ValueFunction(model, rows,
// actions) on the host, one `tobytes()` per row (src/mdp.py:668-669) -- the distinct generating tuples in order of first occurrence,
// their alpha rows (assembled once per tuple, keys accumulated on the way), the byte-dedup of those rows (first position, action of
// the tuple whose last belief comes latest; every key match confirmed bytewise), and only the surviving rows travel back.
extern "C" int pbvi_backup_host_unique(pbvi_model* m, const double* h_beliefs, int nB, const double* h_alphas, int nV, double gamma,
                                       double* h_out_alpha, int out_capacity, int32_t* h_out_action, int* h_n_out, void* stream) {
    PBVI_TRY(check_backup_args(m, h_beliefs, nB, h_alphas, nV, gamma));
    PBVI_REQUIRE(h_n_out != nullptr, "row count output is required");
    *h_n_out = 0;
    if (nB == 0) return PBVI_OK;
    PBVI_REQUIRE(h_out_alpha && h_out_action && out_capacity > 0, "alpha / action outputs with room for out_capacity > 0 rows are required");
    PBVI_CUDA(cudaSetDevice(m->device));
    if (m->hostIn) {      // a previous host call that returned early (an error) may have left copies in flight on the side streams
        PBVI_CUDA(cudaStreamSynchronize(m->hostIn));
        PBVI_CUDA(cudaStreamSynchronize(m->hostOut));
    }
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    m->last_launches = 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (!m->hostIn) {
        PBVI_CUDA(cudaStreamCreateWithFlags(&m->hostIn, cudaStreamNonBlocking));
        PBVI_CUDA(cudaStreamCreateWithFlags(&m->hostOut, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            PBVI_CUDA(cudaEventCreateWithFlags(&m->evIn[i], cudaEventDisableTiming));
            PBVI_CUDA(cudaEventCreateWithFlags(&m->evDone[i], cudaEventDisableTiming));
            PBVI_CUDA(cudaEventCreateWithFlags(&m->evOut[i], cudaEventDisableTiming));
        }
    }
    const size_t S = m->S;
    const int O = m->O, W = 1 + O;
    const int rows = std::min(nB, HOST_CHUNK_ROWS);
    PBVI_TAKE(d_a, double, (size_t)nV * S);
    PBVI_TAKE(d_act, int32_t, (size_t)nB);
    PBVI_TAKE(d_vs, int32_t, (size_t)nB * m->nZ);
    PBVI_TAKE(keys, uint32_t, (size_t)nB * W);
    PBVI_TAKE(first, int32_t, (size_t)nB);
    PBVI_TAKE(last, int32_t, (size_t)nB);
    {   // alphas: straight from page-locked memory, through the pinned staging otherwise
        const size_t bytes = (size_t)nV * S * sizeof(double);
        const void* src = h_alphas;
        if (bytes >= (size_t(8) << 20) && !host_pointer_is_pinned(h_alphas)) {
            void* stage = io_staging(m, bytes);
            if (stage) { parallel_memcpy(stage, h_alphas, bytes); src = stage; }
        }
        PBVI_CUDA(cudaMemcpyAsync(d_a, src, bytes, cudaMemcpyHostToDevice, st));
    }
    int launches = 0;
    bool packed = false;
    PBVI_TRY(host_select_packed(m, h_beliefs, nB, d_a, nV, gamma, d_vs, d_act, st, &launches, &packed));
    const pbvi::Arena::Mark mark = m->arena.mark();
    if (!packed) {
        // dense rows (or a small set): the two-deep chunk pipeline of pbvi_backup_host, upload of chunk k + 1 behind the kernels of chunk k
        double* d_b[2];
        for (int i = 0; i < 2; i++) {
            d_b[i] = m->arena.take<double>((size_t)rows * S);
            if (!d_b[i]) return PBVI_ERR_OOM;
        }
        const pbvi::Arena::Mark inner = m->arena.mark();
        PBVI_CUDA(cudaEventRecord(m->evDone[0], st));
        PBVI_CUDA(cudaStreamWaitEvent(m->hostIn, m->evDone[0], 0));      // the staging is scratch of this call (see pbvi_backup_host)
        for (int lo = 0, k = 0; lo < nB; lo += rows, k++) {
            const int n = std::min(rows, nB - lo), b = k & 1;
            if (k >= 2) PBVI_CUDA(cudaStreamWaitEvent(m->hostIn, m->evDone[b], 0));    // chunk k - 2 has read d_b[b]
            PBVI_CUDA(cudaMemcpyAsync(d_b[b], h_beliefs + (size_t)lo * S, (size_t)n * S * sizeof(double), cudaMemcpyHostToDevice, m->hostIn));
            PBVI_CUDA(cudaEventRecord(m->evIn[b], m->hostIn));
            PBVI_CUDA(cudaStreamWaitEvent(st, m->evIn[b], 0));
            m->arena.rewind(inner);
            m->last_launches = 0;
            PBVI_TRY(select_impl(m, d_b[b], n, d_a, nV, gamma, d_vs + (size_t)lo * m->nZ, nullptr, d_act + lo, st));
            launches += m->last_launches;
            PBVI_CUDA(cudaEventRecord(m->evDone[b], st));
        }
    }
    m->arena.rewind(mark);
    m->last_launches = 0;
    // distinct tuples, in order of first occurrence
    tuple_keys_kernel<<<ceil_div(nB, 256), 256, 0, st>>>(d_vs, d_act, nB, m->A, O, keys);
    int32_t* d_count = nullptr;
    PBVI_TRY(group_keys_impl(m, keys, nB, W, nullptr, first, last, nullptr, &d_count, st));
    int32_t u = 0;
    PBVI_CUDA(cudaMemcpyAsync(&u, d_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    PBVI_REQUIRE(u > 0 && u <= nB, "tuple grouping failed");
    PBVI_TAKE(t_act, int32_t, (size_t)u);
    PBVI_TAKE(t_vsel, int32_t, (size_t)u * O);
    PBVI_TAKE(t_rank, int32_t, (size_t)u);
    tuple_take_kernel<<<ceil_div(u, 256), 256, 0, st>>>(keys, first, last, u, O, t_act, t_vsel, t_rank);
    PBVI_TAKE(d_rows, double, (size_t)u * S);
    PBVI_TAKE(d_hash, uint64_t, (size_t)u * 2);
    PBVI_TRY(assemble_impl(m, d_a, nV, gamma, t_act, t_vsel, (size_t)O, 0, u, d_rows, d_hash, st));
    // byte-dedup of the rows: groups on the 128-bit keys, owner = the tuple whose last belief comes latest
    PBVI_TAKE(gfirst, int32_t, (size_t)u);
    PBVI_TAKE(owner, int32_t, (size_t)u);
    PBVI_TAKE(inverse, int32_t, (size_t)u);
    PBVI_TRY(group_keys_impl(m, reinterpret_cast<const uint32_t*>(d_hash), u, 4, t_rank, gfirst, owner, inverse, &d_count, st));
    int32_t r = 0;
    PBVI_CUDA(cudaMemcpyAsync(&r, d_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    PBVI_REQUIRE(r > 0 && r <= u, "row grouping failed");
    *h_n_out = (int)r;
    m->last_launches += launches + 2;
    if (r > out_capacity) {
        set_error("the backup has %d distinct alpha rows, the output buffers have room for %d", (int)r, out_capacity);
        return PBVI_ERR_BAD_ARG;
    }
    const double* out_rows = d_rows;
    const int32_t* out_act = t_act;
    if (r < u) {
        PBVI_TAKE(mismatch, int32_t, 1);
        PBVI_TRY(confirm_groups_launch(m, d_rows, u, (int)S, gfirst, inverse, mismatch, st));
        int32_t bad = 0;
        PBVI_CUDA(cudaMemcpyAsync(&bad, mismatch, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        PBVI_CUDA(cudaStreamSynchronize(st));
        if (bad) {          // two different rows with one 128-bit key (never observed): the caller falls back to pbvi_backup_host + its own dedup
            set_error("128-bit row keys collided for different alpha rows; use pbvi_backup_host and de-duplicate on the host");
            return PBVI_ERR_UNSUPPORTED;
        }
        PBVI_TAKE(kept, double, (size_t)r * S);
        PBVI_TAKE(kept_act, int32_t, (size_t)r);
        gather_rows_kernel<<<r, 128, 0, st>>>(d_rows, gfirst, (int)S, kept);
        take_int_kernel<<<ceil_div(r, 256), 256, 0, st>>>(t_act, owner, r, kept_act);
        m->last_launches += 2;
        out_rows = kept;
        out_act = kept_act;
    }
    PBVI_CUDA(cudaGetLastError());
    {   // rows: straight into page-locked memory, through the pinned staging otherwise (the alphas left it long ago)
        const size_t bytes = (size_t)r * S * sizeof(double);
        void* stage = (bytes >= (size_t(8) << 20) && !host_pointer_is_pinned(h_out_alpha)) ? io_staging(m, bytes) : nullptr;
        PBVI_CUDA(cudaMemcpyAsync(stage ? stage : (void*)h_out_alpha, out_rows, bytes, cudaMemcpyDeviceToHost, st));
        PBVI_CUDA(cudaMemcpyAsync(h_out_action, out_act, (size_t)r * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        PBVI_CUDA(cudaStreamSynchronize(st));
        if (stage) parallel_memcpy(h_out_alpha, stage, bytes);
    }
    PBVI_CUDA(cudaStreamSynchronize(m->hostIn));
    return PBVI_OK;
}

namespace pbvi {
int max_values_impl(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double* d_max, int32_t* d_arg, cudaStream_t st) {
    return score_argmax(m, d_beliefs, nB, d_alphas, nV, false, d_max, d_arg, st);
}
}  // namespace pbvi

// Sizes the small path accepts: everything of one belief fits in shared memory and the per-belief arithmetic is short.
static bool small_eligible(const pbvi_model* m, int nB, int nV) {
    const double work = (double)nB * nV * m->nZ * m->S;
    return m->S <= 1024 && (size_t)(1 + m->nZ) * m->S + m->A + m->nZ <= 5000 && (long long)nB * m->S <= 262144 && nV <= 4096 &&
           nB <= 16384 && work <= 6e7;
}

extern "C" int pbvi_backup_small_eligible(const pbvi_model* m, int nB, int nV) {
    return (m && nB > 0 && nV > 0 && small_eligible(m, nB, nV)) ? 1 : 0;
}

extern "C" int pbvi_backup_small(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double gamma,
                                 double* d_out_rows, int32_t* h_out_actions, uint64_t* h_out_keys, int* h_n_out, void* stream) {
    PBVI_TRY(check_backup_args(m, d_beliefs, nB, d_alphas, nV, gamma));
    PBVI_REQUIRE(h_n_out != nullptr, "count output is required");
    *h_n_out = 0;
    m->last_launches = 0;
    if (nB == 0) return PBVI_OK;
    PBVI_REQUIRE(d_out_rows && h_out_actions, "row / action outputs are required");
    if (!small_eligible(m, nB, nV)) {
        set_error("pbvi_backup_small: the problem is too large for the single-kernel path (use pbvi_backup_select / pbvi_backup_assemble)");
        return PBVI_ERR_UNSUPPORTED;
    }
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int S = m->S;
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    // one device block [rows | keys | actions] so that a single copy brings everything back; pinned staging of the handle:
    // [rows | keys | actions | gather indices]
    const size_t rowBytes = (size_t)nB * S * sizeof(double), keyBytes = (size_t)nB * 16, actBytes = (size_t)nB * 4;
    PBVI_TAKE(blob, char, rowBytes + keyBytes + actBytes);
    double* rowsAll = reinterpret_cast<double*>(blob);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(blob + rowBytes);
    int32_t* acts = reinterpret_cast<int32_t*>(blob + rowBytes + keyBytes);
    PBVI_TAKE(idx, int32_t, (size_t)nB);
    const size_t need = rowBytes + keyBytes + 2 * actBytes;
    if (m->h_stage_bytes < need) {
        if (m->h_stage) cudaFreeHost(m->h_stage);
        m->h_stage = nullptr;
        m->h_stage_bytes = 0;
        PBVI_CUDA(cudaHostAlloc(&m->h_stage, std::max<size_t>(need, 1 << 16), cudaHostAllocDefault));
        m->h_stage_bytes = std::max<size_t>(need, 1 << 16);
    }
    char* hs = static_cast<char*>(m->h_stage);
    double* hRows = reinterpret_cast<double*>(hs);
    unsigned long long* hKeys = reinterpret_cast<unsigned long long*>(hs + rowBytes);
    int32_t* hActs = reinterpret_cast<int32_t*>(hs + rowBytes + keyBytes);
    int32_t* hIdx = hActs + nB;
    const size_t smem = ((size_t)(1 + m->nZ) * S + m->A) * sizeof(double) + (size_t)m->nZ * sizeof(int);
    small_backup_kernel<<<nB, SMALL_THREADS, smem, st>>>(d_beliefs, d_alphas, m->reachK, m->rtoK, m->rbarT, m->predPtr, m->predK, gamma, S, m->R,
                                                         m->A, m->O, nV, rowsAll, keys, acts);
    PBVI_CUDA(cudaGetLastError());
    PBVI_CUDA(cudaMemcpyAsync(hs, blob, rowBytes + keyBytes + actBytes, cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    // dict semantics of the ValueFunction constructor (src/mdp.py:668-669) over the nB rows: position of the first occurrence, action of
    // the last; open addressing on the 128-bit key, every key match confirmed on the bytes
    int T = 16;
    while (T < 2 * nB) T <<= 1;
    std::vector<int32_t> table((size_t)T, -1);
    int nOut = 0;
    for (int i = 0; i < nB; i++) {
        const unsigned long long k0 = hKeys[(size_t)i * 2], k1 = hKeys[(size_t)i * 2 + 1];
        uint32_t h = (uint32_t)(k0 ^ (k1 >> 17)) & (uint32_t)(T - 1);
        for (;;) {
            const int g = table[h];
            if (g < 0) {
                table[h] = nOut;
                hIdx[nOut] = i;
                h_out_actions[nOut] = hActs[i];
                if (h_out_keys) { h_out_keys[(size_t)nOut * 2] = k0; h_out_keys[(size_t)nOut * 2 + 1] = k1; }
                nOut++;
                break;
            }
            const int f = hIdx[g];
            if (hKeys[(size_t)f * 2] == k0 && hKeys[(size_t)f * 2 + 1] == k1 &&
                std::memcmp(hRows + (size_t)f * S, hRows + (size_t)i * S, (size_t)S * sizeof(double)) == 0) {
                h_out_actions[g] = hActs[i];                     // last action wins
                break;
            }
            h = (h + 1) & (uint32_t)(T - 1);
        }
    }
    PBVI_CUDA(cudaMemcpyAsync(idx, hIdx, (size_t)nOut * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    gather_rows_kernel<<<nOut, 128, 0, st>>>(rowsAll, idx, S, d_out_rows);
    PBVI_CUDA(cudaGetLastError());
    m->last_launches = 2;
    *h_n_out = nOut;
    return PBVI_OK;
}

extern "C" int pbvi_max_values(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double* d_max,
                               int32_t* d_arg, void* stream) {
    PBVI_TRY(check_backup_args(m, d_beliefs, nB, d_alphas, nV, 1.0));
    if (nB == 0) return PBVI_OK;
    PBVI_CUDA(cudaSetDevice(m->device));
    PBVI_TRY(enter_call(m, (cudaStream_t)stream));
    m->last_launches = 0;
    return score_argmax(m, d_beliefs, nB, d_alphas, nV, false, d_max, d_arg, (cudaStream_t)stream);
}
