// Exact LP pruning of alpha vectors (ValueFunction.prune level 3).  The reference meant level 3 to be LP domination (Lark / White
// filter with scipy.optimize.milp, src/mdp.py:834-906); its branch never runs (`pruned_alpha_set` undefined at :872).  Here:
//
//   delta_i = max_{b in simplex} min_{j != i} b . (alpha_i - alpha_j)          (witness margin)
//   tau     = 1e-9 * max(1, max |alpha|)
//
// alpha_i is dropped only with a certificate: a convex combination lambda of other rows with sum_j lambda_j alpha_j[s] > alpha_i[s] + tau
// at every state, re-checked in FP64 from the rows.  Every other row is kept (a witness belief with margin > -tau, a near-tie, a search
// that ran out of budget).  A dropped row lies more than tau below some other row at every belief, so following "the best row that
// beats it" climbs strictly and ends at a kept row: max_v alpha_v . b over the kept rows equals the max over all rows at every belief.
//
// Stages (all FP64):
//   1. row stats + tau           block per row: finite flag and max |alpha|; one block reduces tau
//   2. corner screen             per state the best value, its first row and the runner-up; per row the corner e_s maximising
//                                alpha_i[s] - max_{j != i} alpha_j[s].  A margin > -tau is a witness: the row is kept.
//   3. cutting-plane LP          persistent grid, a block per undecided row.  The block solves the restricted LP over a competitor set J
//                                (max delta s.t. b . (alpha_i - alpha_j) >= delta for j in J, b in the simplex) with a dense revised
//                                simplex (basis inverse in shared memory, pricing over all S columns in parallel), then checks the
//                                verified lower bound m* = min over ALL j of b* . (alpha_i - alpha_j) and the verified upper bound
//                                u = max_s (alpha_i - sum lambda_j alpha_j)[s] from the LP duals; if neither decides, the row that beats
//                                alpha_i most at b* joins J and the LP is solved again.  m* <= delta_i <= delta_J throughout.
//
// Determinism: a row's decision depends only on the rows.  Reductions have a fixed shape with lowest-index tie-breaks; the atomics hand
// out rows to blocks and count outcomes, neither reaches a value.
#include <algorithm>
#include <climits>
#include <cmath>
#include <type_traits>

#include "pbvi_common.cuh"

namespace pbvi {

constexpr int PL_THREADS = 256;
constexpr int J_MAX = 64;                    // competitors of one restricted LP: the basis inverse (J_MAX+1)^2 doubles = 33.8 KB of shared memory
constexpr int M_MAX = J_MAX + 1;             // LP rows: one per competitor + the simplex row
constexpr int PIVOTS_PER_LP = 16 * M_MAX;    // pivot budget of one restricted LP (hitting it leaves the row undecided, i.e. kept)
constexpr int DEGENERATE_RUN = 32;           // consecutive degenerate pivots before the pricing switches to Bland's rule
constexpr double EPS_PRICE = 1e-12;          // reduced-cost and pivot tolerances of the simplex, on rows scaled by 1 / max(1, max|alpha|)
constexpr double EPS_PIVOT = 1e-11;

__device__ __forceinline__ void arg_better(double& v, int& i, double v2, int i2) {
    if (v2 > v || (v2 == v && i2 < i)) { v = v2; i = i2; }
}

// max of (v, i) over the block with the lowest index among equal values; every thread receives the result
__device__ void block_argmax(double& v, int& i, double* sv, int* si) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double v2 = __shfl_down_sync(0xffffffffu, v, off);
        const int i2 = __shfl_down_sync(0xffffffffu, i, off);
        arg_better(v, i, v2, i2);
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { sv[w] = v; si[w] = i; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double bv = sv[0];
        int bi = si[0];
        for (int k = 1; k < PL_THREADS / 32; k++) arg_better(bv, bi, sv[k], si[k]);
        sv[PL_THREADS / 32] = bv;
        si[PL_THREADS / 32] = bi;
    }
    __syncthreads();
    v = sv[PL_THREADS / 32];
    i = si[PL_THREADS / 32];
    __syncthreads();
}

// block per row: finite[i] = every entry finite, rowMax[i] = max |alpha_i| (0 for a non-finite row)
__global__ void __launch_bounds__(PL_THREADS) prune_lp_row_stats_kernel(const double* __restrict__ A, int S, int32_t* __restrict__ finite,
                                                                        double* __restrict__ rowMax) {
    __shared__ double sv[PL_THREADS / 32 + 1];
    __shared__ int si[PL_THREADS / 32 + 1];
    const double* a = A + (size_t)blockIdx.x * S;
    double mx = 0.0;
    int bad = 0;
    for (int s = threadIdx.x; s < S; s += PL_THREADS) {
        const double x = a[s];
        if (!isfinite(x)) bad = 1;
        else mx = fmax(mx, fabs(x));
    }
    bad = __syncthreads_or(bad);
    int dummy = 0;
    block_argmax(mx, dummy, sv, si);
    if (threadIdx.x == 0) {
        finite[blockIdx.x] = bad ? 0 : 1;
        rowMax[blockIdx.x] = bad ? 0.0 : mx;
    }
}

__global__ void __launch_bounds__(PL_THREADS) prune_lp_tau_kernel(const double* __restrict__ rowMax, int n, double* __restrict__ tau) {
    __shared__ double sv[PL_THREADS / 32 + 1];
    __shared__ int si[PL_THREADS / 32 + 1];
    double mx = 0.0;
    for (int i = threadIdx.x; i < n; i += PL_THREADS) mx = fmax(mx, rowMax[i]);
    int dummy = 0;
    block_argmax(mx, dummy, sv, si);
    if (threadIdx.x == 0) tau[0] = 1e-9 * fmax(1.0, mx);
}

// thread per state: best value over the finite rows, its first row, and the runner-up (value and row; equal to the best on a tie)
__global__ void __launch_bounds__(PL_THREADS) prune_lp_columns_kernel(const double* __restrict__ A, int n, int S,
                                                                      const int32_t* __restrict__ finite, double* __restrict__ v1,
                                                                      int32_t* __restrict__ i1, double* __restrict__ v2, int32_t* __restrict__ i2) {
    const int s = blockIdx.x * PL_THREADS + threadIdx.x;
    if (s >= S) return;
    double b1 = -INFINITY, b2 = -INFINITY;
    int j1 = -1, j2 = -1;
    for (int j = 0; j < n; j++) {
        if (!finite[j]) continue;
        const double x = A[(size_t)j * S + s];
        if (j1 < 0 || x > b1) { b2 = b1; j2 = j1; b1 = x; j1 = j; }
        else if (j2 < 0 || x > b2) { b2 = x; j2 = j; }
    }
    v1[s] = b1; i1[s] = j1; v2[s] = b2; i2[s] = j2;
}

// block per row: the best corner.  keep = 1 (witness at a corner, or a non-finite row) or -1 (undecided: goes to the LP, seeded with
// that corner and its best competitor)
__global__ void __launch_bounds__(PL_THREADS) prune_lp_corner_kernel(const double* __restrict__ A, int S, const int32_t* __restrict__ finite,
                                                                     const double* __restrict__ tauP, const double* __restrict__ v1,
                                                                     const int32_t* __restrict__ i1, const double* __restrict__ v2,
                                                                     const int32_t* __restrict__ i2, int32_t* __restrict__ cornerS,
                                                                     int32_t* __restrict__ cornerJ, int32_t* __restrict__ keep,
                                                                     double* __restrict__ bound, int* __restrict__ counts) {
    __shared__ double sv[PL_THREADS / 32 + 1];
    __shared__ int si[PL_THREADS / 32 + 1];
    const int i = blockIdx.x;
    if (!finite[i]) {
        if (threadIdx.x == 0) { keep[i] = 1; bound[i] = NAN; atomicAdd(counts + 0, 1); }
        return;
    }
    const double* a = A + (size_t)i * S;
    double best = -INFINITY;
    int bestS = INT_MAX;
    for (int s = threadIdx.x; s < S; s += PL_THREADS) {
        const bool own = i1[s] == i;
        const int cj = own ? i2[s] : i1[s];
        const double margin = cj < 0 ? INFINITY : a[s] - (own ? v2[s] : v1[s]);
        arg_better(best, bestS, margin, s);
    }
    block_argmax(best, bestS, sv, si);
    if (threadIdx.x == 0) {
        const double tau = tauP[0];
        bound[i] = best;
        if (best > -tau) {
            keep[i] = 1;
            atomicAdd(counts + 0, 1);
        } else {
            keep[i] = -1;
            cornerS[i] = bestS;
            cornerJ[i] = (i1[bestS] == i) ? i2[bestS] : i1[bestS];
        }
    }
}

// residual LP seed, block per row y_i of the pool's first rows: the corner s maximising y_i[s] - max_j x_j[s] (lowest s on a tie), its best
// row of X (pool index off + i1[s]) and that margin, which is m* at b = e_s
__global__ void __launch_bounds__(PL_THREADS) residual_corner_kernel(const double* __restrict__ A, int S, int off, const double* __restrict__ v1,
                                                                     const int32_t* __restrict__ i1, int32_t* __restrict__ cornerS,
                                                                     int32_t* __restrict__ cornerJ, double* __restrict__ bound) {
    __shared__ double sv[PL_THREADS / 32 + 1];
    __shared__ int si[PL_THREADS / 32 + 1];
    const int i = blockIdx.x;
    const double* a = A + (size_t)i * S;
    double best = -INFINITY;
    int bestS = INT_MAX;
    for (int s = threadIdx.x; s < S; s += PL_THREADS) arg_better(best, bestS, a[s] - v1[s], s);
    block_argmax(best, bestS, sv, si);
    if (threadIdx.x == 0) {
        cornerS[i] = bestS;
        cornerJ[i] = off + i1[bestS];
        bound[i] = best;
    }
}

// Cutting-plane LP, a block per undecided row (rows handed out by an atomic counter).  Restricted LP in equality form, rows q < k for the
// competitors J[q], row k the simplex row:
//     sum_s b_s d_q[s] - delta - t_q = 0,   sum_s b_s = 1,   b, t >= 0,   delta free,   maximise delta       (d_q = (alpha_i - alpha_J[q]) / scl)
// Variables: b_s -> id s, t_q -> id S + q, delta -> id S + J_MAX.  delta is basic from the start (at the position of the tightest
// competitor of the seed corner) and, being free, never leaves.  Duals y = row pos(delta) of the basis inverse; at the optimum
// lambda_q = -y_q >= 0 sums to 1 and max_s sum_q lambda_q d_q[s] = delta_J.
// kCert (pbvi_prune_lp_certificates): a pruned row also leaves its certificate, the competitor set J in certIdx[i][0..k) and the weights
// lambda behind the verified bound u in certW[i][0..k) (the rest of the row is left as the caller initialised it).  Nothing else changes.
// The two outputs come as the parameter pack `cert` = (certIdx, certW), empty without kCert: the kernel of pbvi_prune_lp keeps its
// exact parameter list, and with it its code.
__device__ __forceinline__ void write_certificate(int32_t* certIdx, double* certW, int i, int q, int j, double lambda) {
    certIdx[(size_t)i * J_MAX + q] = j;
    certW[(size_t)i * J_MAX + q] = lambda;
}

// Bounded policy iteration (pbvi_bpi_lp) is the instantiation whose pack is one BpiArgs: the restricted master LP of node n over columns
// of a pool, with A = the pool and row i of the pool = W_n of entry i, so the LP code above reads a_i and the columns exactly as it reads
// rows and competitors.  Per launch and entry (keep[i] = -1: active), the column priced at the last tangent belief is checked and
// appended, then one LP is solved from the seed corner; the verified lower bound over all rows is not computed (the pricing is).
struct BpiArgs {
    const int32_t* price;       // [n] pool row of the column priced at bstar (the backup at bstar), -1 on the first launch
    int32_t* cols;              // [n, J_MAX] column lists (pool rows; cols[i][0] = the node's own one-sweep row)
    int32_t* ncols;             // [n] their lengths
    double* bstar;              // [n, S] tangent belief of the last LP (dense)
    double* u;                  // [n] verified bound max_s (W_n - sum_q lambda_q C_q)[s] of the last LP
    double* lambda;             // [n, J_MAX] its weights (0 beyond ncols)
    double* mstar;              // [n] b* . (W_n - C_price) of the last check
};

template <typename... T>
constexpr bool kIsBpi = (false || ... || std::is_same<T, BpiArgs>::value);

__device__ __forceinline__ const BpiArgs& bpi_args(const BpiArgs& a) { return a; }

// The residual LP of incremental pruning (pbvi_ip_residual_lp) is the instantiation whose pack is one ResidualArgs: A is the pool [Y; X]
// (ny rows of the new set, then the nx rows of the old one), the rows i < ny are tested and only X competes.  A row keeps the best
// verified bounds over its LPs -- u (with its J / lambda) and m* (with its b*), both valid for any LP -- and stops when u - m* <= tol.
struct ResidualArgs {
    int off, nx;                // X = pool rows [off, off + nx)
    double tol;                 // stop at u - m* <= tol
    double* u;                  // [ny] verified upper bound on delta_i
    double* mstar;              // [ny] lower bound b* . y_i - max_j b* . x_j
    double* bstar;              // [ny, S] its belief (dense)
    int32_t* certIdx;           // [ny, J_MAX] J of u as rows of X (-1 padded)
    double* certW;              // [ny, J_MAX] lambda of u (0 padded)
    double uBest, mBest;        // per thread: the best bounds of the current row (state kept here, so the other instantiations
                                // declare nothing new and keep their code)
};

template <typename... T>
constexpr bool kIsResidual = (false || ... || std::is_same<T, ResidualArgs>::value);

__device__ __forceinline__ ResidualArgs& residual_args(ResidualArgs& a) { return a; }

// sum of v over the block in a fixed order (warp shuffles, then the warps in order); every thread receives the result
__device__ double block_sum(double v, double* sv) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if ((threadIdx.x & 31) == 0) sv[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = sv[0];
        for (int k = 1; k < PL_THREADS / 32; k++) t += sv[k];
        sv[PL_THREADS / 32] = t;
    }
    __syncthreads();
    const double t = sv[PL_THREADS / 32];
    __syncthreads();
    return t;
}

template <bool kCert, typename... Cert>
__global__ void __launch_bounds__(PL_THREADS, 2) prune_lp_kernel(const double* __restrict__ A, int n, int S, const int32_t* __restrict__ finite,
                                                              const double* __restrict__ tauP, const int32_t* __restrict__ cornerS,
                                                              const int32_t* __restrict__ cornerJ, int32_t* __restrict__ keep,
                                                              double* __restrict__ bound, int* __restrict__ queue, int* __restrict__ counts,
                                                              unsigned long long* __restrict__ stats, Cert... cert) {
    __shared__ double Binv[M_MAX][M_MAX];
    __shared__ double xB[M_MAX], wv[M_MAX], col[M_MAX], prow[M_MAX], lam[J_MAX], suppB[M_MAX];
    __shared__ int basis[M_MAX], J[J_MAX], suppS[M_MAX];
    __shared__ double sv[PL_THREADS / 32 + 1];
    __shared__ int si[PL_THREADS / 32 + 1];
    __shared__ int shRow, shLeave, shNSupp, shJstar, shStatus;
    __shared__ double shScale;
    const int tid = threadIdx.x;
    const double tau = tauP[0];
    const double scl = tau * 1e9, inv = 1.0 / scl;          // = max(1, max|alpha|)
    for (;;) {
        __syncthreads();
        if (tid == 0) shRow = atomicAdd(queue, 1);
        __syncthreads();
        const int i = shRow;
        if (i >= n) return;
        if (keep[i] != -1) continue;
        const double* ai = A + (size_t)i * S;
        const int s0 = cornerS[i];
        if constexpr (!kIsBpi<Cert...>) {
            if (tid == 0) J[0] = cornerJ[i];
        }
        int k = 1;
        int verdict = -1;                                   // 0 pruned, 1 kept by an LP witness, 3 undecided
        double bnd = 0.0;
        unsigned long long pivots = 0, rounds = 0;
        if constexpr (kIsResidual<Cert...>) {
            // the start: m* at the seed corner, u of lambda = e_{J0}; both are valid bounds whatever the LPs below do
            ResidualArgs& g = residual_args(cert...);
            const double* x0 = A + (size_t)cornerJ[i] * S;
            double uv = -INFINITY;
            int us = INT_MAX;
            for (int s = tid; s < S; s += PL_THREADS) {
                arg_better(uv, us, ai[s] - x0[s], s);
                g.bstar[(size_t)i * S + s] = s == s0 ? 1.0 : 0.0;
            }
            block_argmax(uv, us, sv, si);
            g.uBest = uv;
            g.mBest = bound[i];
            if (tid == 0) { g.certIdx[(size_t)i * J_MAX] = cornerJ[i] - g.off; g.certW[(size_t)i * J_MAX] = 1.0; }
            if (g.uBest - g.mBest <= g.tol) verdict = 0;
        }
        if constexpr (kIsBpi<Cert...>) {
            // the column priced at the last b*: m* = b* . (W_n - C_price) <= delta over every column <= delta_J
            const BpiArgs& g = bpi_args(cert...);
            k = g.ncols[i];
            if (tid < k) J[tid] = g.cols[(size_t)i * J_MAX + tid];
            const int p = g.price[i];
            if (p >= 0) {
                double v = 0.0;
                for (int s = tid; s < S; s += PL_THREADS) v = fma(g.bstar[(size_t)i * S + s], ai[s] - A[(size_t)p * S + s], v);
                const double mstar = block_sum(v, sv);
                bool inJ = false;
                for (int q = 0; q < k; q++) inJ |= J[q] == p;
                // 1: not improvable by more than tau, 2: the last LP is optimal, 3: column budget
                const int st = mstar > -tau ? 1 : (inJ || mstar >= bound[i] - tau) ? 2 : k == J_MAX ? 3 : -1;
                if (tid == 0) g.mstar[i] = mstar;
                if (st >= 0) {
                    if (tid == 0) { keep[i] = st; atomicAdd(counts + st, 1); }
                    continue;
                }
                if (tid == 0) { J[k] = p; g.cols[(size_t)i * J_MAX + k] = p; g.ncols[i] = k + 1; }
                k++;
            }
            __syncthreads();
        }
        while (verdict < 0) {
            rounds++;
            const int m = k + 1;
            // ---- cold start at the seed corner: b = e_{s0}, delta = min_q d_q[s0], t_q = d_q[s0] - delta ----
            for (int e = tid; e < M_MAX * M_MAX; e += PL_THREADS) (&Binv[0][0])[e] = 0.0;
            __syncthreads();
            if (tid == 0) {
                int js = 0;
                double dmin = INFINITY;
                for (int q = 0; q < k; q++) {
                    col[q] = (ai[s0] - A[(size_t)J[q] * S + s0]) * inv;
                    if (col[q] < dmin) { dmin = col[q]; js = q; }
                }
                for (int q = 0; q < k; q++) {
                    if (q == js) continue;
                    basis[q] = S + q;
                    Binv[q][q] = -1.0; Binv[q][js] = 1.0; Binv[q][k] = col[q] - col[js];
                    xB[q] = col[q] - col[js];
                }
                basis[js] = S + J_MAX;
                Binv[js][js] = -1.0; Binv[js][k] = col[js];
                xB[js] = col[js];
                basis[k] = s0;
                Binv[k][k] = 1.0;
                xB[k] = 1.0;
                shJstar = js;
                shStatus = 0;
            }
            __syncthreads();
            const int js = shJstar;
            bool bland = false;
            int degenerate = 0, piv = 0;
            // ---- simplex iterations ----
            for (;;) {
                // pricing: reduced cost of b_s is -(sum_q y_q d_q[s] + y_k), of t_q is y_q; basic columns excluded
                double best = -INFINITY;
                int bestId = INT_MAX;
                for (int s = tid; s < S; s += PL_THREADS) {
                    const double x = ai[s];
                    double acc = Binv[js][k];
                    for (int q = 0; q < k; q++) acc = fma(Binv[js][q], (x - A[(size_t)J[q] * S + s]) * inv, acc);
                    const double r = -acc;
                    if (r > EPS_PRICE) {
                        bool basic = false;
                        for (int p = 0; p < m; p++) basic |= basis[p] == s;
                        if (!basic) arg_better(best, bestId, bland ? -(double)s : r, s);
                    }
                }
                if (tid < k) {
                    const double r = Binv[js][tid];
                    if (r > EPS_PRICE) {
                        bool basic = false;
                        for (int p = 0; p < m; p++) basic |= basis[p] == S + tid;
                        if (!basic) arg_better(best, bestId, bland ? -(double)(S + tid) : r, S + tid);
                    }
                }
                block_argmax(best, bestId, sv, si);
                if (bestId == INT_MAX) break;                          // optimal
                if (piv >= PIVOTS_PER_LP) { if (tid == 0) shStatus = 1; __syncthreads(); break; }
                piv++;
                // entering column a and w = Binv a
                const int enter = bestId;
                if (tid <= k) {
                    if (enter < S) col[tid] = tid < k ? (ai[enter] - A[(size_t)J[tid] * S + enter]) * inv : 1.0;
                    else col[tid] = (tid == enter - S) ? -1.0 : 0.0;
                }
                __syncthreads();
                if (tid < m) {
                    double acc = 0.0;
                    for (int q = 0; q < m; q++) acc = fma(Binv[tid][q], col[q], acc);
                    wv[tid] = acc;
                }
                __syncthreads();
                // ratio test (one thread, m <= 65 entries): min x_p / w_p over w_p > 0, delta excluded.  Ties: Bland -> smallest variable
                // id; otherwise the largest pivot, then the lowest position
                if (tid == 0) {
                    int r = -1;
                    double th = INFINITY;
                    for (int p = 0; p < m; p++) {
                        if (p == js || !(wv[p] > EPS_PIVOT)) continue;
                        const double t = fmax(xB[p], 0.0) / wv[p];
                        bool take = r < 0 || t < th;
                        if (!take && t == th) take = bland ? basis[p] < basis[r] : wv[p] > wv[r];
                        if (take) { r = p; th = t; }
                    }
                    shLeave = r;
                    if (r < 0) shStatus = 2;                           // unbounded: cannot happen for a bounded LP, numerical trouble
                    else {
                        degenerate = (th <= 1e-15) ? degenerate + 1 : 0;
                        if (degenerate >= DEGENERATE_RUN) bland = true;
                    }
                }
                __syncthreads();
                const int r = shLeave;
                if (r < 0) break;
                // pivot on (r, enter)
                if (tid < m) prow[tid] = Binv[r][tid] / wv[r];
                __syncthreads();
                for (int e = tid; e < m * m; e += PL_THREADS) {
                    const int p = e / m, q = e - p * m;
                    Binv[p][q] = (p == r) ? prow[q] : fma(-wv[p], prow[q], Binv[p][q]);
                }
                if (tid == 0) {
                    const double xr = fmax(xB[r], 0.0) / wv[r];
                    for (int p = 0; p < m; p++) xB[p] = (p == r) ? xr : fma(-wv[p], xr, xB[p]);
                    basis[r] = enter;
                }
                // bland / degenerate live in thread 0: broadcast
                if (tid == 0) shLeave = bland ? 1 : 0;
                __syncthreads();
                bland = shLeave != 0;
                __syncthreads();
            }
            pivots += piv;
            if (shStatus != 0) { verdict = 3; bnd = NAN; break; }
            // ---- b* (sparse) and lambda ----
            if (tid == 0) {
                int ns = 0;
                double sum = 0.0;
                for (int p = 0; p < m; p++)
                    if (basis[p] < S && xB[p] > 0.0) { suppS[ns] = basis[p]; suppB[ns] = xB[p]; sum += xB[p]; ns++; }
                for (int p = 0; p < ns; p++) suppB[p] /= sum;
                shNSupp = ns;
                double ls = 0.0;
                for (int q = 0; q < k; q++) { lam[q] = fmax(-Binv[js][q], 0.0); ls += lam[q]; }
                shScale = ls;
                for (int q = 0; q < k; q++) lam[q] = ls > 0.0 ? lam[q] / ls : 0.0;
            }
            __syncthreads();
            const int ns = shNSupp;
            // ---- verified lower bound: m* = min over every finite j != i of b* . (alpha_i - alpha_j) ----
            double mv = -INFINITY;
            int mj = INT_MAX;
            if constexpr (kIsResidual<Cert...>) {
                ResidualArgs& g = residual_args(cert...);
                for (int j = g.off + tid; j < g.off + g.nx; j += PL_THREADS) {
                    const double* aj = A + (size_t)j * S;
                    double v = 0.0;
                    for (int p = 0; p < ns; p++) v = fma(suppB[p], ai[suppS[p]] - aj[suppS[p]], v);
                    arg_better(mv, mj, -v, j);
                }
                block_argmax(mv, mj, sv, si);
            } else if constexpr (!kIsBpi<Cert...>) {
                for (int j = tid; j < n; j += PL_THREADS) {
                    if (j == i || !finite[j]) continue;
                    const double* aj = A + (size_t)j * S;
                    double v = 0.0;
                    for (int p = 0; p < ns; p++) v = fma(suppB[p], ai[suppS[p]] - aj[suppS[p]], v);
                    arg_better(mv, mj, -v, j);
                }
                block_argmax(mv, mj, sv, si);
            }
            const double mstar = -mv;
            if constexpr (!kIsBpi<Cert...> && !kIsResidual<Cert...>) {
                if (mstar > -tau) { verdict = 1; bnd = mstar; break; }
            }
            // ---- verified upper bound: u = max_s (alpha_i - sum_q lambda_q alpha_J[q])[s] ----
            double uv = -INFINITY;
            int us = INT_MAX;
            if (shScale > 0.0) {
                for (int s = tid; s < S; s += PL_THREADS) {
                    double c = 0.0;
                    for (int q = 0; q < k; q++) c = fma(lam[q], A[(size_t)J[q] * S + s], c);
                    arg_better(uv, us, ai[s] - c, s);
                }
            } else {
                uv = INFINITY; us = 0;
            }
            block_argmax(uv, us, sv, si);
            if constexpr (kIsBpi<Cert...>) { verdict = 0; bnd = uv; break; }          // one LP per launch: the host prices at b*
            if constexpr (kIsResidual<Cert...>) {
                ResidualArgs& g = residual_args(cert...);
                if (uv < g.uBest) {                          // k only grows: the first k entries replace the previous certificate
                    g.uBest = uv;
                    if (tid < k) { g.certIdx[(size_t)i * J_MAX + tid] = J[tid] - g.off; g.certW[(size_t)i * J_MAX + tid] = lam[tid]; }
                }
                if (mstar > g.mBest) {
                    g.mBest = mstar;
                    double* b = g.bstar + (size_t)i * S;
                    for (int s = tid; s < S; s += PL_THREADS) b[s] = 0.0;
                    __syncthreads();
                    if (tid < ns) b[suppS[tid]] = suppB[tid];
                }
                if (g.uBest - g.mBest <= g.tol) { verdict = 0; break; }
                bool inJ = false;
                for (int q = 0; q < k; q++) inJ |= J[q] == mj;
                if (inJ || k == J_MAX || mj == INT_MAX) { verdict = 3; break; }
                __syncthreads();
                if (tid == 0) J[k] = mj;
                k++;
                __syncthreads();
                continue;
            }
            if (uv < -tau) { verdict = 0; bnd = uv; break; }
            // ---- cut: the row that beats alpha_i most at b* joins J ----
            bool inJ = false;
            for (int q = 0; q < k; q++) inJ |= J[q] == mj;
            if (inJ || k == J_MAX || mj == INT_MAX) { verdict = 3; bnd = mstar; break; }
            __syncthreads();
            if (tid == 0) J[k] = mj;
            k++;
            __syncthreads();
        }
        if constexpr (kCert) {
            if (verdict == 0 && tid < k) write_certificate(cert..., i, tid, J[tid], lam[tid]);   // J and lambda of the LP that gave u
        }
        if constexpr (kIsResidual<Cert...>) {
            ResidualArgs& g = residual_args(cert...);
            if (tid == 0) {
                g.u[i] = g.uBest;
                g.mstar[i] = g.mBest;
                keep[i] = verdict;
                if (verdict != 0) atomicAdd(counts + 3, 1);
                atomicMax(stats + 0, (unsigned long long)k);
                atomicAdd(stats + 1, rounds);
                atomicAdd(stats + 2, pivots);
                atomicAdd(stats + 3, verdict != 0 ? 1ull : 0ull);
            }
            continue;
        }
        if constexpr (kIsBpi<Cert...>) {
            // an LP that ran out of pivots (3) or into numerical trouble (4) leaves the previous LP's outputs as they were
            const BpiArgs& g = bpi_args(cert...);
            if (verdict == 0) {
                double* b = g.bstar + (size_t)i * S;
                for (int s = tid; s < S; s += PL_THREADS) b[s] = 0.0;
                __syncthreads();
                if (tid < shNSupp) b[suppS[tid]] = suppB[tid];
                if (tid < J_MAX) g.lambda[(size_t)i * J_MAX + tid] = tid < k ? lam[tid] : 0.0;
            }
            if (tid == 0) {
                const int st = verdict == 0 ? -1 : shStatus == 1 ? 3 : 4;
                if (verdict == 0) { bound[i] = xB[shJstar] * scl; g.u[i] = bnd; }
                keep[i] = st;
                if (st >= 0) atomicAdd(counts + st, 1);
                atomicMax(stats + 0, (unsigned long long)k);
                atomicAdd(stats + 1, rounds);
                atomicAdd(stats + 2, pivots);
                atomicAdd(stats + 3, 1ull);
            }
            continue;
        }
        if (tid == 0) {
            keep[i] = verdict == 0 ? 0 : 1;
            bound[i] = bnd;
            atomicAdd(counts + (verdict == 0 ? 2 : verdict == 1 ? 1 : 3), 1);
            atomicMax(stats + 0, (unsigned long long)k);
            atomicAdd(stats + 1, rounds);
            atomicAdd(stats + 2, pivots);
            atomicAdd(stats + 3, 1ull);
        }
    }
}

}  // namespace pbvi

using namespace pbvi;

template <bool kCert>
static int prune_lp_impl(pbvi_model* m, const double* d_alphas, int nV, int32_t* d_keep, double* d_bound, int32_t* h_counts,
                         int32_t* d_cert_idx, double* d_cert_w, void* stream) {
    PBVI_REQUIRE(nV >= 0, "nV must be non-negative");
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    if (h_counts) std::fill(h_counts, h_counts + 4, 0);
    m->last_launches = 0;
    std::fill(m->prune_lp_stats, m->prune_lp_stats + 4, 0ll);
    if (nV == 0) return PBVI_OK;
    PBVI_REQUIRE(d_alphas && d_keep, "NULL pointer argument");
    PBVI_REQUIRE(!kCert || (d_cert_idx && d_cert_w), "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, st));
    const int S = m->S, n = nV;
    PBVI_TAKE(finite, int32_t, (size_t)n);
    PBVI_TAKE(rowMax, double, (size_t)n);
    PBVI_TAKE(tau, double, 1);
    PBVI_TAKE(v1, double, (size_t)S);
    PBVI_TAKE(v2, double, (size_t)S);
    PBVI_TAKE(i1, int32_t, (size_t)S);
    PBVI_TAKE(i2, int32_t, (size_t)S);
    PBVI_TAKE(cornerS, int32_t, (size_t)n);
    PBVI_TAKE(cornerJ, int32_t, (size_t)n);
    PBVI_TAKE(counters, int, 8);                          // [0] row queue, [1..4] counts
    PBVI_TAKE(stats, unsigned long long, 4);
    double* bound = d_bound;
    if (!bound) {
        PBVI_TAKE(scratchBound, double, (size_t)n);
        bound = scratchBound;
    }
    PBVI_CUDA(cudaMemsetAsync(counters, 0, 8 * sizeof(int), st));
    PBVI_CUDA(cudaMemsetAsync(stats, 0, 4 * sizeof(unsigned long long), st));
    if (kCert) {
        PBVI_CUDA(cudaMemsetAsync(d_cert_idx, 0xff, (size_t)n * J_MAX * sizeof(int32_t), st));   // -1
        PBVI_CUDA(cudaMemsetAsync(d_cert_w, 0, (size_t)n * J_MAX * sizeof(double), st));
    }
    prune_lp_row_stats_kernel<<<n, PL_THREADS, 0, st>>>(d_alphas, S, finite, rowMax);
    prune_lp_tau_kernel<<<1, PL_THREADS, 0, st>>>(rowMax, n, tau);
    prune_lp_columns_kernel<<<ceil_div(S, PL_THREADS), PL_THREADS, 0, st>>>(d_alphas, n, S, finite, v1, i1, v2, i2);
    prune_lp_corner_kernel<<<n, PL_THREADS, 0, st>>>(d_alphas, S, finite, tau, v1, i1, v2, i2, cornerS, cornerJ, d_keep, bound, counters + 1);
    int perSM = 1;
    if constexpr (kCert) {
        PBVI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, prune_lp_kernel<true, int32_t*, double*>, PL_THREADS, 0));
        const int grid = std::max(1, std::min(n, m->sm_count * std::max(perSM, 1)));
        prune_lp_kernel<true><<<grid, PL_THREADS, 0, st>>>(d_alphas, n, S, finite, tau, cornerS, cornerJ, d_keep, bound, counters, counters + 1,
                                                           stats, d_cert_idx, d_cert_w);
    } else {
        PBVI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, prune_lp_kernel<false>, PL_THREADS, 0));
        const int grid = std::max(1, std::min(n, m->sm_count * std::max(perSM, 1)));
        prune_lp_kernel<false><<<grid, PL_THREADS, 0, st>>>(d_alphas, n, S, finite, tau, cornerS, cornerJ, d_keep, bound, counters, counters + 1,
                                                            stats);
    }
    m->last_launches = 5;
    PBVI_CUDA(cudaGetLastError());
    int32_t c[8];
    unsigned long long sv[4];
    PBVI_CUDA(cudaMemcpyAsync(c, counters, 8 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaMemcpyAsync(sv, stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    if (h_counts) std::copy(c + 1, c + 5, h_counts);
    for (int k = 0; k < 4; k++) m->prune_lp_stats[k] = (long long)sv[k];
    return PBVI_OK;
}

extern "C" int pbvi_prune_lp(pbvi_model* m, const double* d_alphas, int nV, int32_t* d_keep, double* d_bound, int32_t* h_counts, void* stream) {
    return prune_lp_impl<false>(m, d_alphas, nV, d_keep, d_bound, h_counts, nullptr, nullptr, stream);
}

extern "C" int pbvi_prune_lp_certificates(pbvi_model* m, const double* d_alphas, int nV, int32_t* d_keep, double* d_bound, int32_t* h_counts,
                                          int32_t* d_cert_idx, double* d_cert_w, void* stream) {
    return prune_lp_impl<true>(m, d_alphas, nV, d_keep, d_bound, h_counts, d_cert_idx, d_cert_w, stream);
}

extern "C" int pbvi_bpi_lp(pbvi_model* m, const double* d_pool, int nP, int n, double tau, const int32_t* d_corner, const int32_t* d_price,
                           int32_t* d_cols, int32_t* d_ncols, double* d_bstar, double* d_delta, double* d_u, double* d_lambda, double* d_mstar,
                           int32_t* d_status, int64_t* h_stats4, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(n >= 0 && nP >= 2 * n, "need n >= 0 entries and a pool of at least 2n rows (the node rows, then the own columns)");
    PBVI_REQUIRE(tau > 0.0 && std::isfinite(tau), "tau must be finite and > 0");
    if (h_stats4) std::fill(h_stats4, h_stats4 + 4, 0ll);
    m->last_launches = 0;
    if (n == 0) return PBVI_OK;
    PBVI_REQUIRE(d_pool && d_corner && d_price && d_cols && d_ncols && d_bstar && d_delta && d_u && d_lambda && d_mstar && d_status,
                 "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, st));
    PBVI_TAKE(tauD, double, 1);
    PBVI_TAKE(counters, int, 8);                          // [0] entry queue, [1..4] status counts
    PBVI_TAKE(stats, unsigned long long, 4);
    PBVI_CUDA(cudaMemcpyAsync(tauD, &tau, sizeof(double), cudaMemcpyHostToDevice, st));
    PBVI_CUDA(cudaMemsetAsync(counters, 0, 8 * sizeof(int), st));
    PBVI_CUDA(cudaMemsetAsync(stats, 0, 4 * sizeof(unsigned long long), st));
    const BpiArgs args{d_price, d_cols, d_ncols, d_bstar, d_u, d_lambda, d_mstar};
    int perSM = 1;
    PBVI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, prune_lp_kernel<false, BpiArgs>, PL_THREADS, 0));
    const int grid = std::max(1, std::min(n, m->sm_count * std::max(perSM, 1)));
    // finite and cornerJ are not read: no search over rows, and J comes from the entry's column list
    prune_lp_kernel<false><<<grid, PL_THREADS, 0, st>>>(d_pool, n, m->S, nullptr, tauD, d_corner, nullptr, d_status, d_delta, counters,
                                                        counters + 1, stats, args);
    m->last_launches = 1;
    PBVI_CUDA(cudaGetLastError());
    unsigned long long sv[4];
    PBVI_CUDA(cudaMemcpyAsync(sv, stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    if (h_stats4)
        for (int k = 0; k < 4; k++) h_stats4[k] = (long long)sv[k];
    return PBVI_OK;
}

extern "C" int pbvi_ip_residual_lp(pbvi_model* m, const double* d_y, int ny, const double* d_x, int nx, double tau, double* d_u, double* d_mstar,
                                   double* d_bstar, int32_t* d_cert_idx, double* d_cert_w, int64_t* h_stats4, void* stream) {
    PBVI_REQUIRE(m != nullptr, "model handle is NULL");
    PBVI_REQUIRE(ny >= 0 && nx >= 1, "need ny >= 0 rows to test and nx >= 1 rows to test them against");
    PBVI_REQUIRE(tau >= 0.0 && std::isfinite(tau), "tau must be finite and >= 0");
    if (h_stats4) std::fill(h_stats4, h_stats4 + 4, 0ll);
    m->last_launches = 0;
    if (ny == 0) return PBVI_OK;
    PBVI_REQUIRE(d_y && d_x && d_u && d_mstar && d_bstar && d_cert_idx && d_cert_w, "NULL pointer argument");
    PBVI_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    PBVI_TRY(enter_call(m, st));
    const int S = m->S, n = ny + nx;
    PBVI_REQUIRE(n > ny, "ny + nx overflows");
    PBVI_TAKE(pool, double, (size_t)n * S);
    PBVI_TAKE(finite, int32_t, (size_t)n);
    PBVI_TAKE(rowMax, double, (size_t)n);
    PBVI_TAKE(scale, double, 1);
    PBVI_TAKE(v1, double, (size_t)S);
    PBVI_TAKE(v2, double, (size_t)S);
    PBVI_TAKE(i1, int32_t, (size_t)S);
    PBVI_TAKE(i2, int32_t, (size_t)S);
    PBVI_TAKE(cornerS, int32_t, (size_t)ny);
    PBVI_TAKE(cornerJ, int32_t, (size_t)ny);
    PBVI_TAKE(verdict, int32_t, (size_t)ny);
    PBVI_TAKE(bound, double, (size_t)ny);
    PBVI_TAKE(counters, int, 8);                          // [0] row queue, [1..4] counts
    PBVI_TAKE(stats, unsigned long long, 4);
    PBVI_CUDA(cudaMemcpyAsync(pool, d_y, (size_t)ny * S * sizeof(double), cudaMemcpyDeviceToDevice, st));
    PBVI_CUDA(cudaMemcpyAsync(pool + (size_t)ny * S, d_x, (size_t)nx * S * sizeof(double), cudaMemcpyDeviceToDevice, st));
    PBVI_CUDA(cudaMemsetAsync(verdict, 0xff, (size_t)ny * sizeof(int32_t), st));        // -1: every row runs
    PBVI_CUDA(cudaMemsetAsync(counters, 0, 8 * sizeof(int), st));
    PBVI_CUDA(cudaMemsetAsync(stats, 0, 4 * sizeof(unsigned long long), st));
    PBVI_CUDA(cudaMemsetAsync(d_cert_idx, 0xff, (size_t)ny * J_MAX * sizeof(int32_t), st));   // -1
    PBVI_CUDA(cudaMemsetAsync(d_cert_w, 0, (size_t)ny * J_MAX * sizeof(double), st));
    // the simplex works on rows scaled by max(1, max |pool|), as pbvi_prune_lp's does (its tau kernel gives 1e-9 times that)
    prune_lp_row_stats_kernel<<<n, PL_THREADS, 0, st>>>(pool, S, finite, rowMax);
    prune_lp_tau_kernel<<<1, PL_THREADS, 0, st>>>(rowMax, n, scale);
    prune_lp_columns_kernel<<<ceil_div(S, PL_THREADS), PL_THREADS, 0, st>>>(pool + (size_t)ny * S, nx, S, finite + ny, v1, i1, v2, i2);
    residual_corner_kernel<<<ny, PL_THREADS, 0, st>>>(pool, S, ny, v1, i1, cornerS, cornerJ, bound);
    const ResidualArgs args{ny, nx, tau, d_u, d_mstar, d_bstar, d_cert_idx, d_cert_w, INFINITY, -INFINITY};
    int perSM = 1;
    PBVI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, prune_lp_kernel<false, ResidualArgs>, PL_THREADS, 0));
    const int grid = std::max(1, std::min(ny, m->sm_count * std::max(perSM, 1)));
    prune_lp_kernel<false><<<grid, PL_THREADS, 0, st>>>(pool, ny, S, finite, scale, cornerS, cornerJ, verdict, bound, counters, counters + 1,
                                                        stats, args);
    m->last_launches = 5;
    PBVI_CUDA(cudaGetLastError());
    unsigned long long sv[4];
    PBVI_CUDA(cudaMemcpyAsync(sv, stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    PBVI_CUDA(cudaStreamSynchronize(st));
    if (h_stats4)
        for (int k = 0; k < 4; k++) h_stats4[k] = (long long)sv[k];
    return PBVI_OK;
}

extern "C" int pbvi_prune_lp_stats(const pbvi_model* m, int64_t* h_out4) {
    PBVI_REQUIRE(m != nullptr && h_out4 != nullptr, "NULL pointer argument");
    std::copy(m->prune_lp_stats, m->prune_lp_stats + 4, h_out4);
    return PBVI_OK;
}
