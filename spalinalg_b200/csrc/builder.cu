// builder.cu — CooMatrix storage in pinned host memory with the triplets streamed to the device
// while they are pushed (SURVEY.md 8f-4; CooMatrix::push src/coo.rs:431-435, with_capacity
// :162-170, extend :548-574, pop :450-452, clear :470-472).
//
// The reference keeps a Vec<(usize, usize, T)> and hands it to the conversion as a whole.  Done the
// same way here the assembly call starts with 16 + V bytes per triplet over PCIe (C1: 126 MB, 2.4 ms
// against a 0.55 ms sort).  The builder instead keeps the triplets as three pinned SoA arrays
// (row usize, col usize, value) and, every time another CHUNK of them is complete, sends that chunk
// on its own copy stream: two cudaMemcpyAsync of the wide indices into a staging pair followed by
// the narrowing kernel, one cudaMemcpyAsync of the values straight into place.  The host keeps
// pushing while the DMA engine works.  From<&CooMatrix> then only flushes the partial last chunk,
// makes the caller's stream wait on the copy stream's event and runs the device assembly on
// arrays that are already in HBM.
//
// Host state: len (entries pushed), sent (entries handed to the copy stream; positions below it are
// never written by push).  pop()/clear() below `sent` wait for the copy stream and lower `sent`, so
// the positions are sent again when they are refilled.
#include <cstring>
#include <mutex>
#include <new>

#include "kernels.cuh"

using namespace spl;

namespace {
constexpr uint64_t kChunk = 1ull << 19;   // triplets per transfer: 4 MiB per index array
constexpr uint64_t kMinCapacity = 1ull << 12;
}  // namespace

struct spl_coo {
    spl_ctx *copy = nullptr;   // owns the copy stream (and the launch count of the narrowing kernels)
    int dtype = SPL_F64;
    uint64_t nrows = 0, ncols = 0;
    uint64_t len = 0, sent = 0, cap = 0;
    uint64_t *h_row = nullptr, *h_col = nullptr;   // pinned
    unsigned char *h_val = nullptr;                // pinned, cap * vsize
    uint32_t *d_row = nullptr, *d_col = nullptr;   // device, cap
    unsigned char *d_val = nullptr;
    uint64_t *d_wide = nullptr;                    // staging: 2 * kChunk wide indices
    cudaEvent_t landed = nullptr;
    uint64_t counted_launches = 0;                 // launches of `copy` already credited to a caller
    // From<&CooMatrix> takes the builder by shared reference, and the reference's CooMatrix is Sync:
    // two threads may convert the same builder at once.  The conversion's flush of the last partial
    // chunk (send, sent, the staging pair, the landed event) is therefore serialised here.
    std::mutex convert_mu;
    size_t vsize() const { return dtype == SPL_F32 ? 4 : 8; }
};

namespace {

void release(spl_coo *b) {
    if (!b) return;
    if (b->copy) {
        cudaSetDevice(b->copy->device);
        cudaStreamSynchronize(b->copy->stream);
    }
    if (b->h_row) cudaFreeHost(b->h_row);
    if (b->h_col) cudaFreeHost(b->h_col);
    if (b->h_val) cudaFreeHost(b->h_val);
    if (b->d_row) cudaFree(b->d_row);
    if (b->d_col) cudaFree(b->d_col);
    if (b->d_val) cudaFree(b->d_val);
    if (b->d_wide) cudaFree(b->d_wide);
    if (b->landed) cudaEventDestroy(b->landed);
    if (b->copy) spl_ctx_destroy(b->copy);
    delete b;
}

// Grows host and device storage to at least `want` entries (amortised doubling, like Vec).
void reserve(spl_coo *b, uint64_t want) {
    if (want <= b->cap) return;
    uint64_t cap = b->cap ? b->cap : kMinCapacity;
    while (cap < want) cap *= 2;
    const size_t vs = b->vsize();
    uint64_t *hr = nullptr, *hc = nullptr;
    unsigned char *hv = nullptr, *dv = nullptr;
    uint32_t *dr = nullptr, *dc = nullptr;
    try {
        SPL_CUDA(cudaMallocHost(&hr, cap * 8));
        SPL_CUDA(cudaMallocHost(&hc, cap * 8));
        SPL_CUDA(cudaMallocHost(&hv, cap * vs));
        SPL_CUDA(cudaMalloc(&dr, cap * 4));
        SPL_CUDA(cudaMalloc(&dc, cap * 4));
        SPL_CUDA(cudaMalloc(&dv, cap * vs));
        cudaStream_t s = b->copy->stream;
        if (b->sent) {   // what is already on the device moves device to device, behind the copies in flight
            SPL_CUDA(cudaMemcpyAsync(dr, b->d_row, b->sent * 4, cudaMemcpyDeviceToDevice, s));
            SPL_CUDA(cudaMemcpyAsync(dc, b->d_col, b->sent * 4, cudaMemcpyDeviceToDevice, s));
            SPL_CUDA(cudaMemcpyAsync(dv, b->d_val, b->sent * vs, cudaMemcpyDeviceToDevice, s));
        }
        SPL_CUDA(cudaStreamSynchronize(s));   // no transfer reads the old host arrays any more
        if (b->len) {
            std::memcpy(hr, b->h_row, b->len * 8);
            std::memcpy(hc, b->h_col, b->len * 8);
            std::memcpy(hv, b->h_val, b->len * vs);
        }
    } catch (...) {
        if (hr) cudaFreeHost(hr);
        if (hc) cudaFreeHost(hc);
        if (hv) cudaFreeHost(hv);
        if (dr) cudaFree(dr);
        if (dc) cudaFree(dc);
        if (dv) cudaFree(dv);
        throw;
    }
    if (b->h_row) cudaFreeHost(b->h_row);
    if (b->h_col) cudaFreeHost(b->h_col);
    if (b->h_val) cudaFreeHost(b->h_val);
    if (b->d_row) cudaFree(b->d_row);
    if (b->d_col) cudaFree(b->d_col);
    if (b->d_val) cudaFree(b->d_val);
    b->h_row = hr; b->h_col = hc; b->h_val = hv;
    b->d_row = dr; b->d_col = dc; b->d_val = dv;
    b->cap = cap;
}

// Hands entries [sent, upto) to the copy stream, a chunk at a time (the staging pair is reused in
// stream order: the narrowing kernels of one chunk run before the next chunk's copies land).
void send(spl_coo *b, uint64_t upto) {
    cudaStream_t s = b->copy->stream;
    const size_t vs = b->vsize();
    while (b->sent < upto) {
        const uint64_t at = b->sent, n = upto - at < kChunk ? upto - at : kChunk;
        SPL_CUDA(cudaMemcpyAsync(b->d_wide, b->h_row + at, n * 8, cudaMemcpyHostToDevice, s));
        SPL_CUDA(cudaMemcpyAsync(b->d_wide + kChunk, b->h_col + at, n * 8, cudaMemcpyHostToDevice, s));
        SPL_CUDA(cudaMemcpyAsync(b->d_val + at * vs, b->h_val + at * vs, n * vs, cudaMemcpyHostToDevice, s));
        // bounds were asserted on the host at push time; the assembly front checks them again
        narrow_u64(b->copy, b->d_wide, b->d_row + at, n, b->nrows, b->copy->d_scratch);
        narrow_u64(b->copy, b->d_wide + kChunk, b->d_col + at, n, b->ncols, b->copy->d_scratch);
        b->sent = at + n;
    }
}

}  // namespace

#define COO_BEGIN(b)                           \
    if (!(b) || !(b)->copy) return SPL_ERR_ARG; \
    spl_ctx *ctx_ = (b)->copy;                 \
    try {                                      \
        SPL_CUDA(cudaSetDevice(ctx_->device));

#define COO_END                                        \
    }                                                  \
    catch (const spl::Error &e) {                      \
        ctx_->last_error = e.msg;                      \
        return e.status;                               \
    }                                                  \
    catch (...) {                                      \
        ctx_->last_error = "unknown failure";         \
        return SPL_ERR_CUDA;                           \
    }                                                  \
    return SPL_OK;

#pragma GCC visibility push(default)
extern "C" {

int spl_coo_create(spl_ctx *ctx, int dtype, uint64_t nrows, uint64_t ncols, uint64_t capacity,
                   spl_coo **out) {
    if (!ctx || !out) return SPL_ERR_ARG;
    *out = nullptr;
    if (dtype != SPL_F32 && dtype != SPL_F64) {
        ctx->last_error = "Scalar is implemented for f32 and f64 only (src/scalar.rs:55-57)";
        return SPL_ERR_ARG;
    }
    if (nrows == 0 || ncols == 0) {   // CooMatrix::new, src/coo.rs:105-106
        ctx->invalid_reason = nrows == 0 ? 1 : 2;
        ctx->last_error = nrows == 0 ? "nrows must be > 0 (src/coo.rs:105)" : "ncols must be > 0 (src/coo.rs:106)";
        return SPL_ERR_INVALID;
    }
    if (nrows >= (1ull << 32) || ncols >= (1ull << 32)) {
        ctx->last_error = "dimensions must be below 2^32 (device indices are 32 bit)";
        return SPL_ERR_UNSUPPORTED;
    }
    spl_coo *b = new (std::nothrow) spl_coo();
    if (!b) return SPL_ERR_OOM;
    b->dtype = dtype;
    b->nrows = nrows;
    b->ncols = ncols;
    int st = spl_ctx_create(ctx->device, nullptr, &b->copy);
    if (st != SPL_OK) {
        delete b;
        ctx->last_error = "could not create the copy stream";
        return st;
    }
    try {
        SPL_CUDA(cudaSetDevice(ctx->device));
        SPL_CUDA(cudaEventCreateWithFlags(&b->landed, cudaEventDisableTiming));
        SPL_CUDA(cudaMalloc(&b->d_wide, 2 * kChunk * 8));
        reserve(b, capacity ? capacity : kMinCapacity);
    } catch (const spl::Error &e) {
        ctx->last_error = e.msg;
        release(b);
        return e.status;
    }
    *out = b;
    return SPL_OK;
}

int spl_coo_free(spl_coo *b) {
    if (!b) return SPL_ERR_ARG;
    release(b);
    return SPL_OK;
}

const char *spl_coo_last_error(const spl_coo *b) { return b && b->copy ? b->copy->last_error.c_str() : "null builder"; }

int spl_coo_push(spl_coo *b, uint64_t row, uint64_t col, const void *value) {
    if (!b || !b->copy) return SPL_ERR_ARG;
    // the common case touches no CUDA state: bounds, three stores, a counter
    if (value && row < b->nrows && col < b->ncols && b->len < b->cap && b->len + 1 - b->sent < kChunk) {
        b->h_row[b->len] = row;
        b->h_col[b->len] = col;
        std::memcpy(b->h_val + b->len * b->vsize(), value, b->vsize());
        ++b->len;
        return SPL_OK;
    }
    COO_BEGIN(b)
    SPL_REQUIRE(value, SPL_ERR_ARG, "value is NULL");
    SPL_REQUIRE(row < b->nrows, SPL_ERR_ARG, "assertion failed: row < self.nrows (src/coo.rs:432)");
    SPL_REQUIRE(col < b->ncols, SPL_ERR_ARG, "assertion failed: col < self.ncols (src/coo.rs:433)");
    if (b->len == b->cap) reserve(b, b->len + 1);
    b->h_row[b->len] = row;
    b->h_col[b->len] = col;
    std::memcpy(b->h_val + b->len * b->vsize(), value, b->vsize());
    ++b->len;
    if (b->len - b->sent >= kChunk) send(b, b->sent + kChunk);
    COO_END
}

int spl_coo_extend(spl_coo *b, uint64_t len, const uint64_t *row, const uint64_t *col, const void *val) {
    COO_BEGIN(b)
    if (len == 0) return SPL_OK;
    SPL_REQUIRE(row && col && val, SPL_ERR_ARG, "NULL COO array");
    // Extend for CooMatrix (src/coo.rs:566-573) asserts every entry before it stores any
    for (uint64_t i = 0; i < len; ++i) {
        SPL_REQUIRE(row[i] < b->nrows, SPL_ERR_ARG, "assertion failed: *row < self.nrows (src/coo.rs:569)");
        SPL_REQUIRE(col[i] < b->ncols, SPL_ERR_ARG, "assertion failed: *col < self.ncols (src/coo.rs:570)");
    }
    reserve(b, b->len + len);
    const size_t vs = b->vsize();
    // copy chunk-wise so that the first transfers start while the rest is still being copied in
    uint64_t done = 0;
    while (done < len) {
        const uint64_t room = kChunk - (b->len - b->sent) % kChunk;
        const uint64_t n = len - done < room ? len - done : room;
        std::memcpy(b->h_row + b->len, row + done, n * 8);
        std::memcpy(b->h_col + b->len, col + done, n * 8);
        std::memcpy(b->h_val + b->len * vs, (const unsigned char *)val + done * vs, n * vs);
        b->len += n;
        done += n;
        if (b->len - b->sent >= kChunk) send(b, b->sent + kChunk);
    }
    COO_END
}

uint64_t spl_coo_len(const spl_coo *b) { return b ? b->len : 0; }
uint64_t spl_coo_capacity(const spl_coo *b) { return b ? b->cap : 0; }
uint64_t spl_coo_streamed(const spl_coo *b) { return b ? b->sent : 0; }

int spl_coo_reserve(spl_coo *b, uint64_t capacity) {
    COO_BEGIN(b)
    reserve(b, capacity);
    COO_END
}

int spl_coo_truncate(spl_coo *b, uint64_t len) {
    COO_BEGIN(b)
    if (len >= b->len) return SPL_OK;
    if (len < b->sent) {   // the positions will be pushed again: nothing may still be reading them
        SPL_CUDA(cudaStreamSynchronize(b->copy->stream));
        b->sent = len;
    }
    b->len = len;
    COO_END
}

int spl_coo_invalidate(spl_coo *b, uint64_t first) {
    COO_BEGIN(b)
    if (first < b->sent) {   // entries from `first` on were already handed to the copy stream: send them again
        SPL_CUDA(cudaStreamSynchronize(b->copy->stream));
        b->sent = first;
    }
    COO_END
}

int spl_coo_host_ptrs(const spl_coo *b, const uint64_t **row, const uint64_t **col, const void **val) {
    if (!b) return SPL_ERR_ARG;
    if (row) *row = b->h_row;
    if (col) *col = b->h_col;
    if (val) *val = b->h_val;
    return SPL_OK;
}

int spl_mat_from_coo_builder(spl_ctx *ctx, spl_coo *b, int format, int dedup, int dropzero, spl_mat **out) {
    if (!ctx || !b || !b->copy || !out) return SPL_ERR_ARG;
    *out = nullptr;
    try {
        SPL_REQUIRE(format == SPL_CSR || format == SPL_CSC, SPL_ERR_ARG, "unknown format");
        SPL_REQUIRE(ctx->device == b->copy->device, SPL_ERR_ARG, "builder lives on another device");
        SPL_CUDA(cudaSetDevice(ctx->device));
        ctx->pdl_chain = false;
        {
            std::lock_guard<std::mutex> lock(b->convert_mu);
            send(b, b->len);   // the partial last chunk
            SPL_CUDA(cudaEventRecord(b->landed, b->copy->stream));
            SPL_CUDA(cudaStreamWaitEvent(ctx->stream, b->landed, 0));
            ctx->launches += b->copy->launches - b->counted_launches;
            b->counted_launches = b->copy->launches;
        }
        *out = assemble_from_coo_any(ctx, format, b->dtype, (uint32_t)b->nrows, (uint32_t)b->ncols, b->len,
                                     b->d_row, b->d_col, b->d_val, dedup, dropzero);
        publish_mat(ctx, *out);
    } catch (const spl::Error &e) {
        ctx->last_error = e.msg;
        return e.status;
    } catch (...) {
        ctx->last_error = "unknown failure";
        return SPL_ERR_CUDA;
    }
    return SPL_OK;
}

}  // extern "C"
#pragma GCC visibility pop
