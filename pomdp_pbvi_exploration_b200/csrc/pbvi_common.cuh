// Shared declarations for the PBVI B200 engine: model handle, scratch arena, error plumbing.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/pbvi_b200.h"

namespace pbvi {

// ---- tiling constants of the score kernel (see score_kernel.cuh) --------------------------------
#ifndef PBVI_KC
#define PBVI_KC 4
#endif
constexpr int KC = PBVI_KC;         // source states per K chunk -- the sparsity-skipping granule along K (4, 8 or 16).  On the bench workload
                               // a 16-state granule executes 1.46x the flops of an 8-state one (tools/sparsity_analysis.py)
#ifndef PBVI_SUB
#define PBVI_SUB 4
#endif
constexpr int SUB = PBVI_SUB;  // chunks per pipeline stage of the score kernel: zeros are skipped per KC-state chunk, the mbarrier handshake
                               // is paid per SUB chunks (a dense workload runs like a kernel with SUB*KC-state chunks)
constexpr int SKC = SUB * KC;  // source states per stage
constexpr int BM = 64;         // beliefs per block tile
constexpr int BN = 256;        // alpha vectors per block tile
constexpr int RG = 16;         // beliefs per row group (one warp's rows) -- the skipping granule along M
constexpr int NRG = BM / RG;   // 4 row groups per tile
constexpr int SCORE_THREADS = NRG * (BN / 64) * 32;   // consumer threads of the score kernel (+ one producer warp)

// d_signs[SIGN_DENSE]: some alpha of the running select / max_values call is NaN or +-inf.  Every zero-skipping rule of the engine rests
// on "0 * x = 0", which fails for non-finite x (the reference's NumPy arithmetic yields NaN there), so all of them are switched off
// for such a call and the dense product is computed.
constexpr int SIGN_DENSE = 6;

void set_error(const char* fmt, ...);

#define PBVI_CUDA(call)                                                                              \
    do {                                                                                             \
        cudaError_t _e = (call);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            pbvi::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return (_e == cudaErrorMemoryAllocation) ? PBVI_ERR_OOM : PBVI_ERR_CUDA;                 \
        }                                                                                            \
    } while (0)

#define PBVI_REQUIRE(cond, msg)                                          \
    do {                                                                 \
        if (!(cond)) {                                                   \
            pbvi::set_error("bad argument: %s (%s)", msg, #cond);        \
            return PBVI_ERR_BAD_ARG;                                     \
        }                                                                \
    } while (0)

#define PBVI_TRY(expr)                \
    do {                              \
        int _rc = (expr);             \
        if (_rc != PBVI_OK) return _rc; \
    } while (0)

// Grow-only device scratch owned by the model handle.  Allocation is a bump pointer over a list of chunks; a call that
// outgrows the current chunk adds one (pointers handed out earlier stay valid), and the next `reset()` -- the start of
// the next API call -- consolidates them, so steady-state calls never allocate.
struct Arena {
    struct Chunk { char* base; size_t cap, off; };
    std::vector<Chunk> chunks;
    void* take_bytes(size_t bytes);     // nullptr (and the error string set) when the device is out of memory
    void reset();
    // scratch of a sub-step of one call: everything taken after mark() is handed back by rewind() (the kernels that used it precede the
    // next user in stream order)
    struct Mark { size_t chunks, off; };
    Mark mark() const { return Mark{chunks.size(), chunks.empty() ? 0 : chunks.back().off}; }
    void rewind(const Mark& k) {
        for (size_t i = k.chunks; i < chunks.size(); i++) chunks[i].off = 0;
        if (k.chunks > 0 && k.chunks <= chunks.size()) chunks[k.chunks - 1].off = k.off;
    }
    void release();
    template <typename T> T* take(size_t n) { return reinterpret_cast<T*>(take_bytes(n * sizeof(T))); }
    static size_t padded(size_t bytes) { return (bytes + 255) & ~size_t(255); }
};

#define PBVI_TAKE(var, T, n)                         \
    T* var = m->arena.take<T>(n);                    \
    if (!var) return PBVI_ERR_OOM

// 128-bit row key = two independent NH hashes (the almost-universal hash of UMAC) over the 8-byte words of the row:
//     h_j = sum_i (lo(w_i) + k_{j,0}(i)) * (hi(w_i) + k_{j,1}(i))     32-bit wrapping adds, 32x32 -> 64-bit product, sum mod 2^64
// with four 32-bit position keys per word index drawn from splitmix64 (row_key_words), finalised with the row length.  Wrapping
// addition makes the value independent of the reduction shape (shuffles, shared memory, atomics).  A word costs one wide
// multiply per hash once its keys are at hand: the assemble kernel, which computes the key of a row while writing it, loads the
// keys of its states from a per-model table once per block instead of running the mixer per element.  Every key match is
// confirmed bytewise before rows are merged, so the key only has to make false matches rare, not impossible.
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {   // splitmix64 finaliser
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27; x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}
__host__ __device__ __forceinline__ uint4 row_key_words(int i) {
    const uint64_t a = mix64(0x9e3779b97f4a7c15ull * (uint64_t)(2 * (int64_t)i + 1));
    const uint64_t b = mix64(0xc2b2ae3d27d4eb4full * (uint64_t)(2 * (int64_t)i + 2) + 0xd6e8feb86659fd93ull);
    return make_uint4((uint32_t)a, (uint32_t)(a >> 32), (uint32_t)b, (uint32_t)(b >> 32));
}
__host__ __device__ __forceinline__ uint64_t row_hash_term0(uint64_t w, const uint4& k) {
    return (uint64_t)((uint32_t)w + k.x) * (uint64_t)((uint32_t)(w >> 32) + k.y);
}
__host__ __device__ __forceinline__ uint64_t row_hash_term1(uint64_t w, const uint4& k) {
    return (uint64_t)((uint32_t)w + k.z) * (uint64_t)((uint32_t)(w >> 32) + k.w);
}
__host__ __device__ __forceinline__ uint64_t row_hash_final0(uint64_t a, int rowLen) { return mix64(a + (uint64_t)rowLen); }
__host__ __device__ __forceinline__ uint64_t row_hash_final1(uint64_t b, int rowLen) { return mix64(b ^ (uint64_t)rowLen); }

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t ceil_div_sz(size_t a, size_t b) { return (a + b - 1) / b; }

}  // namespace pbvi

struct pbvi_model {
    int S = 0, A = 0, O = 0, R = 0;
    int K = 0;        // S*R
    int Sp = 0;       // S padded to a multiple of KC
    int nChunks = 0;  // Sp / KC
    int nZ = 0;       // A*O
    int device = 0;
    int sm_count = 148;
    bool has_probs = false;

    // action-major device tables
    int32_t* reachK = nullptr;   // [A][S*R]      landing state of k = s*R + r
    double* rtoK = nullptr;      // [A][O][S*R]   RTO
    double* probK = nullptr;     // [A][S*R]      transition probabilities (nullptr when not supplied)
    double* rbarT = nullptr;     // [A][S]
    // CSR of the non-zero expected rewards per action (b . Rbar[:,a] touches only these)
    int32_t* rbarNzPtr = nullptr;  // [A+1]
    int32_t* rbarNzIdx = nullptr;  // [nnz] state
    double* rbarNzVal = nullptr;   // [nnz]
    // R == 1 fast path of the score kernel: chunk-padded copies (pad: landing state 0, RTO 0)
    int32_t* reachP = nullptr;   // [A][Sp]
    double* rtoP = nullptr;      // [A][O][Sp]
    uint8_t* zMask = nullptr;    // [nZ][nChunks]  1 iff some RTO[s,a,o,:] != 0 for a source state s of the chunk
    int32_t* zOrder = nullptr;   // [nZ] (a*O+o) sorted by decreasing number of live chunks (heavy blocks first)
    // CSR over landing states (bincount order of Belief.update)
    int32_t* predPtr = nullptr;  // [A][S+1]
    int32_t* predK = nullptr;    // [A][K]       source k's in ascending order
    // NumPy pairwise-sum tree over a length-S row
    int2* pwLeaves = nullptr;    // [nLeaves] (offset, length)
    int2* pwNodes = nullptr;     // [nNodes]  (left, right); child >= 0: node id, < 0: leaf ~id; root is the last node
    int32_t* pwLevelNodes = nullptr;   // [nNodes] node ids grouped by tree level (children always in an earlier level)
    int32_t* pwLevelPtr = nullptr;     // [nLevels + 1]
    int nLevels = 0;
    bool no_chain_kernel = false;      // pbvi_set_option("chain_kernel", 0): belief chains as one launch per step-kernel (tests, A/B)
    int chain_mode = 2;                // 2 (default): a cluster of 8 blocks; 1: one persistent block (pbvi_set_option("chain_kernel", ...))
    uint4* hashKeys = nullptr;   // [S] row_key_words(s): position keys of the 128-bit row key
    int nLeaves = 0, nNodes = 0;

    pbvi::Arena arena;
    // stream guard: the scratch arena, the sign flags and the tile counter are reused by consecutive calls IN STREAM ORDER; a call that
    // arrives on another stream than its predecessor first waits (on the device) for everything the predecessor enqueued
    cudaStream_t last_stream = nullptr;
    bool has_last_stream = false;
    cudaEvent_t evGuard = nullptr;
    void* h_stage = nullptr;     // pinned host staging of pbvi_backup_small (grow-only)
    size_t h_stage_bytes = 0;
    // instrumentation of the last select / max_values call
    unsigned long long* d_stats = nullptr;   // [1] live (tile, z, chunk, row group) quadruples visited by the score launch
    // sign information for the exact-zero shortcut of the value pass: with RTO, Rbar, every belief and every alpha >= 0 a sum
    // that comes out exactly 0 consists of zero terms only, so the reference-order value is exactly 0 as well
    bool model_nonneg = false;               // RTO >= 0 and Rbar >= 0 (checked once on the host)
    const uint8_t* last_bits = nullptr;      // belief occupancy bits of the running select call (arena memory)
    int* d_signs = nullptr;                  // [8] ([4]: tile queue counter of the score kernel) set by the last select: [0] some alpha < 0 or NaN, [1] some belief < 0 or NaN,
                                             //     [SIGN_DENSE] some alpha NaN or +-inf; [3] the same for the alphas of the last assemble call
    double last_dense_flops = 0.0;
    double last_exec_scale = 0.0;            // flops per visited quadruple
    int last_launches = 0;
    // optional timing of the dominant (score) kernel with CUDA events on the caller's stream
    bool profile = false;
    bool score_timed = false;
    cudaEvent_t evScore0 = nullptr, evScore1 = nullptr;
    // pbvi_backup_host: upload / download streams and the events of its two-deep chunk pipeline (created on first use)
    cudaStream_t hostIn = nullptr, hostOut = nullptr;
    cudaEvent_t evIn[2] = {nullptr, nullptr}, evDone[2] = {nullptr, nullptr}, evOut[2] = {nullptr, nullptr};
    void* h_pack = nullptr;      // pinned staging of the packed belief upload of pbvi_backup_host_unique (grow-only)
    size_t h_pack_bytes = 0;
    void* h_io = nullptr;        // pinned staging for pageable alpha / output buffers of the same call (grow-only)
    size_t h_io_bytes = 0;
    long long prune_lp_stats[4] = {0, 0, 0, 0};   // last pbvi_prune_lp: largest |J|, restricted LPs solved, simplex pivots, rows sent to the LP
};

namespace pbvi {
// implemented in backup.cu, used by other translation units
int transpose_alphas(pbvi_model* m, const double* d_alphas, int nV, int Vp, double* d_alphaT, cudaStream_t st);
// per-device function attributes (dynamic shared memory opt-ins) of each translation unit; pbvi_model_create calls them with the
// handle's device current, so a second handle on another GPU of the same process is configured too
// building blocks shared across translation units (none of them resets the arena: the calling entry point does)
int belief_successors_impl(pbvi_model* m, const double* d_beliefs, int n, int normalise, double* d_out, double* d_norm, cudaStream_t st);
int row_hash_launch(pbvi_model* m, const double* d_rows, int n, int row_len, uint64_t* d_hash, cudaStream_t st);
int max_values_impl(pbvi_model* m, const double* d_beliefs, int nB, const double* d_alphas, int nV, double* d_max, int32_t* d_arg, cudaStream_t st);
// start of an API call that uses the handle's scratch: stream guard (see pbvi_model::last_stream) + arena rewind
int enter_call(pbvi_model* m, cudaStream_t st);
int unpack_rows_launch(pbvi_model* m, const uint32_t* d_bitmap, const int32_t* d_row_start, const double* d_packed, int n, int row_len,
                       int slab_rows, long long region_chunks, double* d_out, cudaStream_t st);
int group_keys_impl(pbvi_model* m, const uint32_t* d_keys, int n, int words, const int32_t* d_rank, int32_t* d_first, int32_t* d_last,
                    int32_t* d_inverse, int32_t** d_count_out, cudaStream_t st);
int confirm_groups_launch(pbvi_model* m, const double* d_rows, int n, int row_len, const int32_t* d_first, const int32_t* d_inverse,
                          int32_t* d_mismatch, cudaStream_t st);
int configure_backup_kernels();
int configure_belief_kernels();
int configure_misc_kernels();
}
