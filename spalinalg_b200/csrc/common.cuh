// common.cuh — context, matrix handle, error plumbing and small device helpers
// shared by every translation unit of libspalinalg_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/spl.h"

namespace spl {

struct Error {
    int status;
    std::string msg;
};

#define SPL_CUDA(expr)                                                                   \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            throw ::spl::Error{_e == cudaErrorMemoryAllocation ? SPL_ERR_OOM : SPL_ERR_CUDA, \
                               std::string(#expr) + ": " + cudaGetErrorString(_e)};      \
        }                                                                                \
    } while (0)

#define SPL_REQUIRE(cond, status, text)                      \
    do {                                                     \
        if (!(cond)) throw ::spl::Error{(status), (text)};   \
    } while (0)

constexpr int kNumSmFallback = 148;
// 32-bit positions: kernels step a position by up to a tile (<= 65536 entries) past the last entry
// before testing it, so entry counts stay that far below 2^32.
constexpr uint64_t kMaxEntries = (1ull << 32) - 65536;
// longest row whose column offsets the SpMV plan keeps as the matrix's row pattern (spl_mat::pattern_off)
constexpr uint32_t kPatternMax = 64;

// A test-only setting from the environment: true and *v when `name` holds a decimal number and nothing else;
// false when it is unset, empty or anything else, so that a typo leaves the library's default in place.
inline bool env_u64(const char *name, unsigned long long *v) {
    const char *s = std::getenv(name);
    if (!s || *s < '0' || *s > '9') return false;
    char *end = nullptr;
    *v = std::strtoull(s, &end, 10);        // ULLONG_MAX on overflow: clamped by the callers
    return *end == '\0';
}

}  // namespace spl

// Opaque handles of the C ABI.
struct spl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    int num_sms = spl::kNumSmFallback;
    std::string last_error;
    int invalid_reason = 0;
    uint64_t launches = 0;
    uint32_t *h_scratch = nullptr;   // pinned, 64 words: small device->host read-backs
    uint32_t *d_scratch = nullptr;   // device, 64 words
    // host-vector SpMV pipeline (spl_spmv_host): upload and download streams and the events that
    // order them against the compute stream; created on first use
    static constexpr int kPipeChunks = 8;
    cudaStream_t up_stream = nullptr, down_stream = nullptr;
    cudaEvent_t pipe_ev[2 * kPipeChunks + 2] = {};
    // programmatic dependent launch: true while the last thing this context put on its stream was a
    // stream-kernel SpMV (whose CTAs signal launch_dependents); the next one may then start its
    // matrix prefetch under the tail of that product.  Any other entry point clears it.
    // the library's own stream-ordered memory pool on this device (shared by all contexts of the
    // process): freed blocks stay in it for the next call without touching the device's default
    // pool, which other libraries in the process (torch) allocate from
    cudaMemPool_t pool = nullptr;
    bool pdl_chain = false;
    bool pdl_prev = false;     // pdl_chain as the current entry point found it
};

struct spl_mat {
    int format = SPL_CSR;
    int dtype = SPL_F64;
    uint32_t nrows = 0, ncols = 0, nnz = 0;
    uint32_t *ptr = nullptr;   // nmajor + 1
    uint32_t *ind = nullptr;   // nnz
    void *val = nullptr;       // nnz * sizeof(T)
    // "wide" matrices (2^32 - 65536 stored entries or more): 64-bit positions.  ptr64 replaces ptr (which
    // stays NULL), nnz64 holds the count and nnz is pinned to 0xffffffff; only the kernels in wide.cu
    // (validation, SpMV, transpose / convert, download, entry chunks) take them.
    uint64_t *ptr64 = nullptr;
    uint64_t nnz64 = 0;
    bool wide() const { return ptr64 != nullptr; }
    uint64_t entries() const { return ptr64 ? nnz64 : (uint64_t)nnz; }
    // SpMV plan (filled lazily by the first spl_spmv on this matrix; read-only afterwards).
    // A matrix may be shared read-only by several host threads / contexts (spl.h): the first
    // caller plans under plan_mu, everybody else sees plan_ready (acquire) and only reads.
    std::mutex plan_mu;
    std::atomic<int> plan_ready{0};
    int plan_kernel = 0;       // SPL_SPMV_VECTOR / SPL_SPMV_MERGE
    int plan_lanes = 0;        // lanes per row of the vector kernel
    uint32_t max_row_len = 0;
    uint32_t col_min = 0, col_max = 0;   // smallest / largest stored column (plan; meaningless when nnz == 0)
    uint32_t *merge_rows = nullptr;   // merge-path tile start rows (merge_tiles + 1)
    uint32_t merge_tiles = 0;
    uint32_t *split_rows = nullptr;   // nnz-split kernel: row holding the first entry of each chunk
    uint32_t split_chunks = 0;
    // hot-column cache (skewed matrices whose few hottest columns carry much of the matrix):
    // col_order[j] = the j-th most frequent column (hot_count of them); ind_rank = the matrix's
    // column indices with every hot column replaced by (flag | its slot j)
    uint32_t *ind_rank = nullptr;
    uint32_t *col_order = nullptr;
    uint32_t hot_count = 0;
    std::atomic<int> hot_state{0};    // 0 not tried, 1 one split product done, 2 decided (ind_rank set or not)
    double hot_coverage = 0.0;        // share of the stored entries that fall in the hot columns
    // sliced copy for the vector-class SpMV (regular rows): slices of 32 consecutive rows stored
    // column-major inside the slice (entry k of the 32 rows contiguous), padded to the slice's
    // longest row.  slice_ptr[s] = sum of the widths of the slices before s (offset = 32 * that).
    uint32_t *slice_ptr = nullptr;
    uint32_t *slice_ind = nullptr;
    void *slice_val = nullptr;
    uint64_t slice_entries = 0;       // padded entries stored
    // host-vector SpMV pipeline: row chunks and, per chunk, how long a prefix of x its rows need
    // (1 + the largest column index in the chunks up to it); pipe_state 0 = not planned yet
    uint32_t pipe_rows[spl_ctx::kPipeChunks + 1] = {};
    uint32_t pipe_need[spl_ctx::kPipeChunks] = {};
    std::atomic<int> pipe_state{0};
    std::atomic<int> slice_state{0};  // 0 not tried, 1 one vector product done, 2 decided (slice_ptr set or not)
    // stream kernel (persistent, TMA-pipelined; regular rows): tiles of stream_rows consecutive rows,
    // stream_cap = shared-memory stage capacity in entries (0: a window of stream_rows rows does not fit:
    // kernel not usable).  For a grid of stream_grid CTAs: stream_cta_rows[b] = first row of CTA b (ranges
    // balanced on rows + stored entries), stream_xhi[b * stream_max_tiles + k] = 1 + the largest column of
    // CTA b's tile k (0 if it has no entry), stream_xlo0[b] = smallest column of its first tile: the
    // producer prefetches the leading edge of x into L2 from them; stream_tile_lo = position of every
    // tile's first stored entry (same layout, one more slot per CTA)
    uint32_t *stream_cta_rows = nullptr, *stream_xhi = nullptr, *stream_xlo0 = nullptr, *stream_tile_lo = nullptr;
    uint32_t stream_rows = 0, stream_cap = 0, stream_grid = 0, stream_max_tiles = 0;
    // row pattern (plan; depends on ptr and ind only): pattern_len = K = max_row_len when 0 < K <= kPatternMax and
    // some row r at or after nrows / 2 has K entries; pattern_off[j] = ind[ptr[r] + j] - r (mod 2^32) for the first
    // such r (a shard's local matrix: local rows, global columns, offsets shifted by its first row).  A stream
    // tile is regular when each of its rows r has K entries at columns r + pattern_off[j]: the stream kernel
    // then fetches its values only.  stream_tile_reg[slot] = 1 for a regular tile (layout of stream_tile_lo),
    // stream_regular = how many tiles of the grid are regular.
    uint32_t pattern_off[spl::kPatternMax] = {};
    uint32_t pattern_len = 0;
    uint32_t *stream_tile_reg = nullptr;
    uint32_t stream_regular = 0;

    // CSR form of a CSC matrix (same matrix, other format), built by the first product y = A x on it
    // and kept: products on a CscMatrix then run the row kernels at full speed and in the reference's
    // summation order.  Owned by this matrix; dropped when the values change.
    std::atomic<spl_mat *> twin{nullptr};
    // Sharing across contexts (spl.h: a matrix may be used read-only by several host threads, each
    // with its own context and stream).  `home` is the stream the matrix was created on and `ready`
    // the event recorded there behind the last kernel that wrote it: a context on another stream
    // waits on it before its first use.  Every use from another stream leaves an event in `foreign`
    // (one slot per stream), so that whoever frees the matrix waits for those readers first.
    cudaStream_t home = nullptr;
    cudaEvent_t ready = nullptr;
    std::mutex use_mu;
    struct ForeignUse { cudaStream_t stream; cudaEvent_t done; };
    std::vector<ForeignUse> foreign;

    uint32_t nmajor() const { return format == SPL_CSR ? nrows : ncols; }
    uint32_t nminor() const { return format == SPL_CSR ? ncols : nrows; }
    size_t vsize() const { return dtype == SPL_F32 ? 4 : 8; }
};

namespace spl {

// Stream-ordered device allocation (pool-backed: freed blocks are reused without a sync).
template <typename T>
inline T *dalloc(spl_ctx *ctx, size_t count) {
    void *p = nullptr;
    size_t bytes = (count ? count : 1) * sizeof(T);
    SPL_CUDA(cudaMallocFromPoolAsync(&p, bytes, ctx->pool, ctx->stream));
    return static_cast<T *>(p);
}
inline void *dalloc_bytes(spl_ctx *ctx, size_t bytes) {
    void *p = nullptr;
    SPL_CUDA(cudaMallocFromPoolAsync(&p, bytes ? bytes : 1, ctx->pool, ctx->stream));
    return p;
}
inline void dfree(spl_ctx *ctx, void *p) {
    if (p) cudaFreeAsync(p, ctx->stream);
}

// RAII temporary: freed (stream-ordered) when it goes out of scope, also on exceptions.
template <typename T>
struct Tmp {
    spl_ctx *ctx;
    T *p;
    Tmp(spl_ctx *c, size_t count) : ctx(c), p(dalloc<T>(c, count)) {}
    ~Tmp() { dfree(ctx, p); }
    Tmp(const Tmp &) = delete;
    Tmp &operator=(const Tmp &) = delete;
    T *release() { T *q = p; p = nullptr; return q; }
    operator T *() const { return p; }
};

inline void count_launch(spl_ctx *ctx, int n = 1) { ctx->launches += (uint64_t)n; }

inline void check_launch(spl_ctx *ctx, const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) throw Error{SPL_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e)};
    count_launch(ctx);
}

// Reads `words` (<= 64) uint32 from device memory to the host, synchronising the stream.
inline void read_back(spl_ctx *ctx, const uint32_t *d_src, uint32_t *dst, int words) {
    SPL_CUDA(cudaMemcpyAsync(ctx->h_scratch, d_src, sizeof(uint32_t) * words, cudaMemcpyDeviceToHost,
                             ctx->stream));
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < words; ++i) dst[i] = ctx->h_scratch[i];
}

inline int bits_for(uint64_t count) {   // bits needed to represent values in [0, count)
    int b = 0;
    while (b < 64 && (count - 1) >> b) ++b;
    return count <= 1 ? 0 : b;
}

inline unsigned div_up(uint64_t a, uint64_t b) { return (unsigned)((a + b - 1) / b); }

// ---------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Inclusive warp scan (shuffle up).
__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane_id() >= (unsigned)o) v += t;
    }
    return v;
}

// Block-wide exclusive scan of one uint32 per thread.  `warp_sums` is shared memory with at
// least blockDim.x/32 + 1 slots.  Returns the exclusive prefix; *total gets the block sum.
// Contains two __syncthreads(); every thread of the block must call it.
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t *warp_sums,
                                                         uint32_t *total) {
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    uint32_t incl = warp_inclusive_scan(v);
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t s = lane < nwarps ? warp_sums[lane] : 0u;
        uint32_t si = warp_inclusive_scan(s);
        if (lane < nwarps) warp_sums[lane] = si - s;
        if (lane == 31) warp_sums[nwarps] = si;
    }
    __syncthreads();
    uint32_t res = warp_sums[warp] + incl - v;
    if (total) *total = warp_sums[nwarps];
    return res;
}

// first index in [lo, hi) with a[idx] > key  (a non-decreasing)
__device__ __forceinline__ uint32_t upper_bound_u32(const uint32_t *__restrict__ a, uint32_t lo,
                                                    uint32_t hi, uint32_t key) {
    while (lo < hi) {
        uint32_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(a + mid) <= key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// first index in [lo, hi) with a[idx] > key  (a non-decreasing), 64-bit positions
__device__ __forceinline__ uint64_t upper_bound_u64(const uint64_t *__restrict__ a, uint64_t lo, uint64_t hi,
                                                    uint64_t key) {
    while (lo < hi) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(a + mid) <= key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// Streaming load (SASS LDG.E.NA, L1::no_allocate) for data a kernel reads exactly once with fully
// coalesced warps — the col/val stream of the nnz-split and merge SpMV kernels — so that it does
// not push the reusable x out of L1.  Measured on B200 (profiles/r1_spmv_notes.md): +6 % on the
// R-MAT matrix; NOT for the vector kernel, whose few-lanes-per-row loads re-read their sectors
// from L1 (0.88 -> 0.41 of peak on 9-entry rows when its stream bypassed L1).
__device__ __forceinline__ uint32_t ld_stream(const uint32_t *p) {
    uint32_t v;
    asm("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_stream(const float *p) {
    float v;
    asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double ld_stream(const double *p) {
    double v;
    asm("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

struct NoPayload {};

// Marks a freshly created matrix complete on the creating context's stream.
inline void publish_mat(spl_ctx *ctx, spl_mat *m) {
    if (!m) return;
    m->home = ctx->stream;
    if (!m->ready) SPL_CUDA(cudaEventCreateWithFlags(&m->ready, cudaEventDisableTiming));
    SPL_CUDA(cudaEventRecord(m->ready, ctx->stream));
}

// Scope of one use of a matrix by a context: a context on the matrix's home stream is ordered by
// the stream itself; any other context waits for `ready` first and leaves an event behind.
struct MatUse {
    spl_ctx *ctx;
    spl_mat *m;
    bool foreign = false;
    MatUse(spl_ctx *c, const spl_mat *mat) : ctx(c), m(const_cast<spl_mat *>(mat)) {
        if (!m || !m->ready || m->home == ctx->stream) return;
        foreign = true;
        SPL_CUDA(cudaStreamWaitEvent(ctx->stream, m->ready, 0));
    }
    ~MatUse() {
        if (!foreign) return;
        std::lock_guard<std::mutex> lock(m->use_mu);
        for (auto &f : m->foreign)
            if (f.stream == ctx->stream) { cudaEventRecord(f.done, ctx->stream); return; }
        cudaEvent_t e = nullptr;
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return; }
        cudaEventRecord(e, ctx->stream);
        m->foreign.push_back({ctx->stream, e});
    }
    MatUse(const MatUse &) = delete;
    MatUse &operator=(const MatUse &) = delete;
};

// Rust's unary minus on floats is a sign-bit flip for every input, NaN included (the GPU's FNEG
// path may canonicalise NaN), so negate on the integer view.
__device__ __forceinline__ float flip_sign(float v) {
    return __uint_as_float(__float_as_uint(v) ^ 0x80000000u);
}
__device__ __forceinline__ double flip_sign(double v) {
    return __longlong_as_double(__double_as_longlong(v) ^ (long long)0x8000000000000000ull);
}

}  // namespace spl
