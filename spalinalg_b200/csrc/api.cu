// api.cu — the extern "C" boundary declared in include/spl.h.  Plain pointers and sizes in,
// status codes out; nothing unwinds across it.  No CPU fallback: every entry point needs a
// live CUDA context.
#include <algorithm>
#include <cstring>
#include <mutex>
#include <new>
#include <string>

#include "kernels.cuh"

using namespace spl;

#define API_BEGIN(ctx)                         \
    if (!(ctx)) return SPL_ERR_ARG;            \
    try {                                      \
        (ctx)->pdl_prev = (ctx)->pdl_chain;    \
        (ctx)->pdl_chain = false;              \
        SPL_CUDA(cudaSetDevice((ctx)->device));

#define API_END(ctx)                                   \
    }                                                  \
    catch (const spl::Error &e) {                      \
        (ctx)->last_error = e.msg;                     \
        return e.status;                               \
    }                                                  \
    catch (const std::bad_alloc &) {                   \
        (ctx)->last_error = "host allocation failed"; \
        return SPL_ERR_OOM;                            \
    }                                                  \
    catch (...) {                                      \
        (ctx)->last_error = "unknown failure";        \
        return SPL_ERR_CUDA;                           \
    }                                                  \
    return SPL_OK;

namespace {

void check_enums(int format, int dtype) {
    SPL_REQUIRE(format == SPL_CSR || format == SPL_CSC, SPL_ERR_ARG, "unknown format");
    SPL_REQUIRE(dtype == SPL_F32 || dtype == SPL_F64, SPL_ERR_ARG,
                "Scalar is implemented for f32 and f64 only (src/scalar.rs:55-57)");
}

void check_dims(spl_ctx *ctx, uint64_t nrows, uint64_t ncols) {
    if (nrows == 0) {
        ctx->invalid_reason = 1;
        throw Error{SPL_ERR_INVALID, "nrows must be > 0 (src/csr.rs:144, src/coo.rs:105)"};
    }
    if (ncols == 0) {
        ctx->invalid_reason = 2;
        throw Error{SPL_ERR_INVALID, "ncols must be > 0 (src/csr.rs:145, src/coo.rs:106)"};
    }
    SPL_REQUIRE(nrows < (1ull << 32) && ncols < (1ull << 32), SPL_ERR_UNSUPPORTED,
                "dimensions must be below 2^32 (device indices are 32 bit)");
}

// One private memory pool per device for the whole library.  Freed blocks stay in it (release
// threshold raised on THIS pool only), so the temporaries of the next call are reused without a
// synchronisation; the device's default pool, which torch and others allocate from, is left alone.
cudaMemPool_t library_pool(int device) {
    static std::mutex mu;
    static cudaMemPool_t pools[64] = {};
    std::lock_guard<std::mutex> lock(mu);
    SPL_REQUIRE(device >= 0 && device < 64, SPL_ERR_ARG, "device ordinal out of range");
    if (!pools[device]) {
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        cudaMemPool_t pool = nullptr;
        SPL_CUDA(cudaMemPoolCreate(&pool, &props));
        uint64_t threshold = UINT64_MAX;
        SPL_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold));
        pools[device] = pool;
    }
    return pools[device];
}

[[noreturn]] void invalid(spl_ctx *ctx, int reason, const char *text) {
    ctx->invalid_reason = reason;
    throw Error{SPL_ERR_INVALID, text};
}

void require_narrow(const spl_mat *m, const char *what) {
    if (m && m->wide())
        throw Error{SPL_ERR_UNSUPPORTED, std::string(what) + ": operand has 2^32 - 65536 stored entries or more (64-bit "
                    "positions); supported on such matrices: new / validation, SpMV, transpose, CSR<->CSC, download, iter"};
}

const char *kReasonText[10] = {
    "",
    "nrows must be > 0",
    "ncols must be > 0",
    "ptr.len() != n + 1",
    "ptr[0] != 0",
    "ind.len() != ptr[n]",
    "values.len() != ptr[n]",
    "ptr is not sorted",
    "index out of range",
    "indices not strictly increasing inside a row/column",
};

}  // namespace

#pragma GCC visibility push(default)
extern "C" {

int spl_ctx_create(int device, void *stream, spl_ctx **out) {
    if (!out) return SPL_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
        cudaGetLastError();
        return SPL_ERR_CUDA;   // no device, no product path: there is no CPU fallback
    }
    spl_ctx *ctx = new (std::nothrow) spl_ctx();
    if (!ctx) return SPL_ERR_OOM;
    ctx->device = device;
    try {
        SPL_CUDA(cudaSetDevice(device));
        if (stream) {
            ctx->stream = static_cast<cudaStream_t>(stream);
        } else {
            SPL_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
            ctx->owns_stream = true;
        }
        int sms = 0;
        SPL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        ctx->num_sms = sms > 0 ? sms : kNumSmFallback;
        ctx->pool = library_pool(device);
        SPL_CUDA(cudaMallocHost(&ctx->h_scratch, 64 * sizeof(uint32_t)));
        SPL_CUDA(cudaMalloc(&ctx->d_scratch, 64 * sizeof(uint32_t)));
        SPL_CUDA(cudaMemset(ctx->d_scratch, 0, 64 * sizeof(uint32_t)));
    } catch (const spl::Error &) {
        if (ctx->h_scratch) cudaFreeHost(ctx->h_scratch);
        if (ctx->d_scratch) cudaFree(ctx->d_scratch);
        if (ctx->owns_stream) cudaStreamDestroy(ctx->stream);
        delete ctx;
        return SPL_ERR_CUDA;
    }
    *out = ctx;
    return SPL_OK;
}

int spl_ctx_destroy(spl_ctx *ctx) {
    if (!ctx) return SPL_ERR_ARG;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->h_scratch) cudaFreeHost(ctx->h_scratch);
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    for (cudaEvent_t e : ctx->pipe_ev)
        if (e) cudaEventDestroy(e);
    if (ctx->up_stream) cudaStreamDestroy(ctx->up_stream);
    if (ctx->down_stream) cudaStreamDestroy(ctx->down_stream);
    if (ctx->owns_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return SPL_OK;
}

int spl_ctx_sync(spl_ctx *ctx) {
    API_BEGIN(ctx)
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    API_END(ctx)
}

// page-locked host memory: no context, plain status codes
int spl_host_alloc(uint64_t bytes, void **out) {
    if (!out) return SPL_ERR_ARG;
    *out = nullptr;
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? (size_t)bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        return SPL_ERR_CUDA;
    }
    *out = p;
    return SPL_OK;
}
int spl_host_free(void *p) {
    if (!p) return SPL_OK;
    if (cudaFreeHost(p) != cudaSuccess) { cudaGetLastError(); return SPL_ERR_CUDA; }
    return SPL_OK;
}
int spl_host_register(void *p, uint64_t bytes) {
    if (!p || !bytes) return SPL_ERR_ARG;
    if (cudaHostRegister(p, (size_t)bytes, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); return SPL_ERR_CUDA; }
    return SPL_OK;
}
int spl_host_unregister(void *p) {
    if (!p) return SPL_OK;
    if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return SPL_ERR_CUDA; }
    return SPL_OK;
}

int spl_ctx_trim(spl_ctx *ctx) {
    API_BEGIN(ctx)
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    SPL_CUDA(cudaMemPoolTrimTo(ctx->pool, 0));          // freed blocks the library's pool still holds go back to the driver
    API_END(ctx)
}

const char *spl_last_error(const spl_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
int spl_invalid_reason(const spl_ctx *ctx) { return ctx ? ctx->invalid_reason : 0; }
uint64_t spl_launch_count(const spl_ctx *ctx) { return ctx ? ctx->launches : 0; }

int spl_mat_from_coo_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                         uint64_t len, const uint32_t *row_dev, const uint32_t *col_dev,
                         const void *val_dev, int dedup, int dropzero, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(out, SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    check_enums(format, dtype);
    check_dims(ctx, nrows, ncols);
    SPL_REQUIRE(len == 0 || (row_dev && col_dev && val_dev), SPL_ERR_ARG, "NULL COO array");
    *out = assemble_from_coo_any(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, len, row_dev, col_dev,
                                 val_dev, dedup, dropzero);
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_mat_from_coo(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                     uint64_t len, const uint64_t *row, const uint64_t *col, const void *val,
                     int dedup, int dropzero, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(out, SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    check_enums(format, dtype);
    check_dims(ctx, nrows, ncols);
    SPL_REQUIRE(len == 0 || (row && col && val), SPL_ERR_ARG, "NULL COO array");
    const size_t vs = dtype == SPL_F32 ? 4 : 8;
    Tmp<uint32_t> r32(ctx, len), c32(ctx, len);
    Tmp<unsigned char> v(ctx, len * vs);
    if (assemble_is_bucketed(len)) {       // long lists: the indices narrow through a fixed staging buffer
        constexpr uint64_t kChunk = 1ull << 26;
        Tmp<uint64_t> stage(ctx, std::min(kChunk, len));
        SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, sizeof(uint32_t), ctx->stream));
        for (uint64_t at = 0; at < len; at += kChunk) {
            const uint64_t cnt = std::min(kChunk, len - at);
            SPL_CUDA(cudaMemcpyAsync(stage, row + at, cnt * 8, cudaMemcpyHostToDevice, ctx->stream));
            narrow_u64(ctx, stage, r32 + at, cnt, nrows, ctx->d_scratch);
            SPL_CUDA(cudaMemcpyAsync(stage, col + at, cnt * 8, cudaMemcpyHostToDevice, ctx->stream));
            narrow_u64(ctx, stage, c32 + at, cnt, ncols, ctx->d_scratch);
        }
        SPL_CUDA(cudaMemcpyAsync(v, val, len * vs, cudaMemcpyHostToDevice, ctx->stream));
    } else if (len) {
        Tmp<uint64_t> wide(ctx, len);
        SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, sizeof(uint32_t), ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(wide, row, len * 8, cudaMemcpyHostToDevice, ctx->stream));
        narrow_u64(ctx, wide, r32, len, nrows, ctx->d_scratch);
        SPL_CUDA(cudaMemcpyAsync(wide, col, len * 8, cudaMemcpyHostToDevice, ctx->stream));
        narrow_u64(ctx, wide, c32, len, ncols, ctx->d_scratch);
        SPL_CUDA(cudaMemcpyAsync(v, val, len * vs, cudaMemcpyHostToDevice, ctx->stream));
    }
    // bounds (CooMatrix::push, src/coo.rs:432-433) are re-checked on the narrowed arrays
    *out = assemble_from_coo_any(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, len, r32, c32, v, dedup,
                                 dropzero);
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_mat_from_compressed_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                                uint64_t nnz, const uint32_t *ptr_dev, const uint32_t *ind_dev,
                                const void *val_dev, int validate, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(out, SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    check_enums(format, dtype);
    check_dims(ctx, nrows, ncols);
    SPL_REQUIRE(nnz < kMaxEntries, SPL_ERR_UNSUPPORTED, "nnz must be below 2^32 - 65536");
    SPL_REQUIRE(ptr_dev && (nnz == 0 || (ind_dev && val_dev)), SPL_ERR_ARG, "NULL array");
    const uint32_t nmajor = (uint32_t)(format == SPL_CSR ? nrows : ncols);
    const uint32_t nminor = (uint32_t)(format == SPL_CSR ? ncols : nrows);
    if (validate) {
        uint32_t first = 0, last = 0;
        read_back(ctx, ptr_dev, &first, 1);
        read_back(ctx, ptr_dev + nmajor, &last, 1);
        if (first != 0) invalid(ctx, 4, kReasonText[4]);
        if (last != nnz) invalid(ctx, 5, kReasonText[5]);
        int why = validate_compressed(ctx, nmajor, nminor, (uint32_t)nnz, ptr_dev, ind_dev);
        if (why) invalid(ctx, why, kReasonText[why]);
    }
    spl_mat *m = new_mat(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, (uint32_t)nnz);
    try {
        SPL_CUDA(cudaMemcpyAsync(m->ptr, ptr_dev, ((size_t)nmajor + 1) * 4, cudaMemcpyDeviceToDevice,
                                 ctx->stream));
        if (nnz) {
            SPL_CUDA(cudaMemcpyAsync(m->ind, ind_dev, nnz * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            SPL_CUDA(cudaMemcpyAsync(m->val, val_dev, nnz * m->vsize(), cudaMemcpyDeviceToDevice,
                                     ctx->stream));
        }
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    *out = m;
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_mat_from_compressed(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                            uint64_t ptr_len, const uint64_t *ptr, uint64_t ind_len,
                            const uint64_t *ind, uint64_t val_len, const void *val, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(out, SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    check_enums(format, dtype);
    check_dims(ctx, nrows, ncols);                                     // assertions 1, 2
    const uint64_t nmajor = format == SPL_CSR ? nrows : ncols;
    const uint64_t nminor = format == SPL_CSR ? ncols : nrows;
    if (ptr_len != nmajor + 1) invalid(ctx, 3, kReasonText[3]);
    SPL_REQUIRE(ptr, SPL_ERR_ARG, "ptr is NULL");
    if (ptr[0] != 0) invalid(ctx, 4, kReasonText[4]);
    if (ind_len != ptr[nmajor]) invalid(ctx, 5, kReasonText[5]);
    if (val_len != ptr[nmajor]) invalid(ctx, 6, kReasonText[6]);
    const uint64_t nnz = ind_len;
    SPL_REQUIRE(nnz == 0 || (ind && val), SPL_ERR_ARG, "NULL array");
    if (nnz >= wide_min_nnz()) {           // 64-bit positions: the pointers go up as they are, the indices narrow in chunks
        spl_mat *w = new_wide_mat(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, nnz);
        try {
            SPL_CUDA(cudaMemcpyAsync(w->ptr64, ptr, (nmajor + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
            constexpr uint64_t kChunk = 1ull << 26;
            Tmp<uint64_t> stage(ctx, kChunk);
            SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, 2 * sizeof(uint32_t), ctx->stream));
            for (uint64_t at = 0; at < nnz; at += kChunk) {
                const uint64_t cnt = std::min(kChunk, nnz - at);
                SPL_CUDA(cudaMemcpyAsync(stage, ind + at, cnt * 8, cudaMemcpyHostToDevice, ctx->stream));
                narrow_u64(ctx, stage, w->ind + at, cnt, nminor, ctx->d_scratch + 1);
            }
            SPL_CUDA(cudaMemcpyAsync(w->val, val, nnz * w->vsize(), cudaMemcpyHostToDevice, ctx->stream));
            uint32_t flags[2] = {0, 0};
            read_back(ctx, ctx->d_scratch, flags, 2);
            int why = wide_validate(ctx, w);
            if (why == 0 && flags[1]) why = 8;
            if (why) invalid(ctx, why, kReasonText[why]);
        } catch (...) {
            free_mat(ctx, w);
            throw;
        }
        *out = w;
        publish_mat(ctx, *out);
        return SPL_OK;
    }

    spl_mat *m = new_mat(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, (uint32_t)nnz);
    try {
        {
            Tmp<uint64_t> wide(ctx, nmajor + 1 > nnz ? nmajor + 1 : nnz);
            SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, 2 * sizeof(uint32_t), ctx->stream));
            SPL_CUDA(cudaMemcpyAsync(wide, ptr, (nmajor + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
            narrow_u64(ctx, wide, m->ptr, nmajor + 1, nnz + 1, ctx->d_scratch);       // flag word 0
            if (nnz) {
                SPL_CUDA(cudaMemcpyAsync(wide, ind, nnz * 8, cudaMemcpyHostToDevice, ctx->stream));
                narrow_u64(ctx, wide, m->ind, nnz, nminor, ctx->d_scratch + 1);       // flag word 1
                SPL_CUDA(cudaMemcpyAsync(m->val, val, nnz * m->vsize(), cudaMemcpyHostToDevice,
                                         ctx->stream));
            }
        }
        uint32_t flags[2] = {0, 0};
        read_back(ctx, ctx->d_scratch, flags, 2);
        // a pointer above nnz cannot be part of a sorted array ending in nnz  -> assertion 7
        if (flags[0]) invalid(ctx, 7, kReasonText[7]);
        int why = validate_compressed(ctx, (uint32_t)nmajor, (uint32_t)nminor, (uint32_t)nnz, m->ptr,
                                      m->ind);
        if (why == 0 && flags[1]) why = 8;
        if (why) invalid(ctx, why, kReasonText[why]);
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    *out = m;
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_mat_from_compressed_dev64(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                                  uint64_t nnz, const uint64_t *ptr_dev, const uint32_t *ind_dev,
                                  const void *val_dev, int validate, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(out, SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    check_enums(format, dtype);
    check_dims(ctx, nrows, ncols);
    SPL_REQUIRE(ptr_dev && (nnz == 0 || (ind_dev && val_dev)), SPL_ERR_ARG, "NULL array");
    const uint32_t nmajor = (uint32_t)(format == SPL_CSR ? nrows : ncols);
    const uint32_t nminor = (uint32_t)(format == SPL_CSR ? ncols : nrows);
    uint32_t ends[4] = {0, 0, 0, 0};                     // ptr[0] and ptr[n] as two 32-bit words each
    if (validate) {
        read_back(ctx, reinterpret_cast<const uint32_t *>(ptr_dev), ends, 2);
        read_back(ctx, reinterpret_cast<const uint32_t *>(ptr_dev + nmajor), ends + 2, 2);
        if (ends[0] != 0 || ends[1] != 0) invalid(ctx, 4, kReasonText[4]);
        if ((((uint64_t)ends[3] << 32) | ends[2]) != nnz) invalid(ctx, 5, kReasonText[5]);
    }
    if (nnz < wide_min_nnz()) {                          // fits 32-bit positions: the usual matrix
        spl_mat *m = new_mat(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, (uint32_t)nnz);
        try {
            SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, sizeof(uint32_t), ctx->stream));
            narrow_u64(ctx, ptr_dev, m->ptr, (size_t)nmajor + 1, nnz + 1, ctx->d_scratch);
            if (nnz) {
                SPL_CUDA(cudaMemcpyAsync(m->ind, ind_dev, nnz * 4, cudaMemcpyDeviceToDevice, ctx->stream));
                SPL_CUDA(cudaMemcpyAsync(m->val, val_dev, nnz * m->vsize(), cudaMemcpyDeviceToDevice, ctx->stream));
            }
            if (validate) {
                uint32_t over = 0;
                read_back(ctx, ctx->d_scratch, &over, 1);
                if (over) invalid(ctx, 7, kReasonText[7]);
                int why = validate_compressed(ctx, nmajor, nminor, (uint32_t)nnz, m->ptr, m->ind);
                if (why) invalid(ctx, why, kReasonText[why]);
            }
        } catch (...) {
            free_mat(ctx, m);
            throw;
        }
        *out = m;
    } else {
        spl_mat *m = new_wide_mat(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, nnz);
        try {
            SPL_CUDA(cudaMemcpyAsync(m->ptr64, ptr_dev, ((size_t)nmajor + 1) * 8, cudaMemcpyDeviceToDevice, ctx->stream));
            SPL_CUDA(cudaMemcpyAsync(m->ind, ind_dev, nnz * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            SPL_CUDA(cudaMemcpyAsync(m->val, val_dev, nnz * m->vsize(), cudaMemcpyDeviceToDevice, ctx->stream));
            if (validate) {
                int why = wide_validate(ctx, m);
                if (why) invalid(ctx, why, kReasonText[why]);
            }
        } catch (...) {
            free_mat(ctx, m);
            throw;
        }
        *out = m;
    }
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_mat_eye(spl_ctx *ctx, int format, int dtype, uint64_t size, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(out, SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    check_enums(format, dtype);
    check_dims(ctx, size, size);   // assert!(size > 0), src/csr.rs:180
    spl_mat *m = new_mat(ctx, format, dtype, (uint32_t)size, (uint32_t)size, (uint32_t)size);
    try {
        fill_eye(ctx, dtype, (uint32_t)size, m->ptr, m->ind, m->val);
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    *out = m;
    publish_mat(ctx, *out);
    API_END(ctx)
}

static spl_mat *regroup(spl_ctx *ctx, const spl_mat *in, int out_format, uint32_t out_rows,
                        uint32_t out_cols) {
    if (in->wide()) return wide_regroup(ctx, in, out_format, out_rows, out_cols);
    // out's major axis is in's minor axis
    spl_mat *m = new_mat(ctx, out_format, in->dtype, out_rows, out_cols, in->nnz);
    try {
        recompress(ctx, in->dtype, in->nmajor(), in->nminor(), in->nnz, in->ptr, in->ind, in->val,
                   m->ptr, m->ind, m->val);
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    return m;
}

int spl_mat_convert(spl_ctx *ctx, const spl_mat *in, int format, spl_mat **out) {
    API_BEGIN(ctx)
    MatUse use_in(ctx, in);
    SPL_REQUIRE(in && out, SPL_ERR_ARG, "NULL handle");
    *out = nullptr;
    check_enums(format, in->dtype);
    if (format == in->format && in->wide()) {
        spl_mat *m = new_wide_mat(ctx, in->format, in->dtype, in->nrows, in->ncols, in->nnz64);
        SPL_CUDA(cudaMemcpyAsync(m->ptr64, in->ptr64, ((size_t)in->nmajor() + 1) * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(m->ind, in->ind, (size_t)in->nnz64 * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(m->val, in->val, (size_t)in->nnz64 * in->vsize(), cudaMemcpyDeviceToDevice, ctx->stream));
        *out = m;
        publish_mat(ctx, *out);
    } else if (format == in->format) {
        spl_mat *m = new_mat(ctx, in->format, in->dtype, in->nrows, in->ncols, in->nnz);
        SPL_CUDA(cudaMemcpyAsync(m->ptr, in->ptr, ((size_t)in->nmajor() + 1) * 4,
                                 cudaMemcpyDeviceToDevice, ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(m->ind, in->ind, (size_t)in->nnz * 4, cudaMemcpyDeviceToDevice,
                                 ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(m->val, in->val, (size_t)in->nnz * in->vsize(),
                                 cudaMemcpyDeviceToDevice, ctx->stream));
        *out = m;
        publish_mat(ctx, *out);
    } else {
        *out = regroup(ctx, in, format, in->nrows, in->ncols);
        publish_mat(ctx, *out);   // same matrix, other format
    }
    API_END(ctx)
}

int spl_mat_transpose(spl_ctx *ctx, const spl_mat *in, spl_mat **out) {
    API_BEGIN(ctx)
    MatUse use_in(ctx, in);
    SPL_REQUIRE(in && out, SPL_ERR_ARG, "NULL handle");
    *out = nullptr;
    *out = regroup(ctx, in, in->format, in->ncols, in->nrows);
    publish_mat(ctx, *out);   // same format, dims swapped
    API_END(ctx)
}

int spl_mat_add(spl_ctx *ctx, const spl_mat *a, const spl_mat *b, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(a && b && out, SPL_ERR_ARG, "NULL handle");
    *out = nullptr;
    require_narrow(a, "spl_mat_add");
    require_narrow(b, "spl_mat_add");
    MatUse use_a(ctx, a);
    MatUse use_b(ctx, b);
    *out = addsub(ctx, a, b, 0);
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_mat_sub(spl_ctx *ctx, const spl_mat *a, const spl_mat *b, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(a && b && out, SPL_ERR_ARG, "NULL handle");
    *out = nullptr;
    require_narrow(a, "spl_mat_sub");
    require_narrow(b, "spl_mat_sub");
    MatUse use_a(ctx, a);
    MatUse use_b(ctx, b);
    *out = addsub(ctx, a, b, 1);
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_mat_mul(spl_ctx *ctx, const spl_mat *a, const spl_mat *b, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(a && b && out, SPL_ERR_ARG, "NULL handle");
    *out = nullptr;
    require_narrow(a, "spl_mat_mul");
    require_narrow(b, "spl_mat_mul");
    MatUse use_a(ctx, a);
    MatUse use_b(ctx, b);
    *out = spgemm(ctx, a, b);
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_mat_neg(spl_ctx *ctx, const spl_mat *a, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(a && out, SPL_ERR_ARG, "NULL handle");
    *out = nullptr;
    require_narrow(a, "spl_mat_neg");
    MatUse use_a(ctx, a);
    spl_mat *m = new_mat(ctx, a->format, a->dtype, a->nrows, a->ncols, a->nnz);
    try {
        SPL_CUDA(cudaMemcpyAsync(m->ptr, a->ptr, ((size_t)a->nmajor() + 1) * 4,
                                 cudaMemcpyDeviceToDevice, ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(m->ind, a->ind, (size_t)a->nnz * 4, cudaMemcpyDeviceToDevice,
                                 ctx->stream));
        negate(ctx, a->dtype, a->nnz, a->val, m->val);
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    *out = m;
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_spmv_ex(spl_ctx *ctx, const spl_mat *a, const void *x_dev, void *y_dev, int kernel) {
    API_BEGIN(ctx)
    MatUse use_a(ctx, a);
    SPL_REQUIRE(a && x_dev && y_dev, SPL_ERR_ARG, "NULL argument");
    if (a->wide()) wide_spmv(ctx, a, x_dev, y_dev);          // 64-bit positions: the vector kernel of wide.cu
    else spmv(ctx, a, x_dev, y_dev, kernel & 0xff, (kernel >> 8) & 0xff);
    API_END(ctx)
}

int spl_spmv(spl_ctx *ctx, const spl_mat *a, const void *x_dev, void *y_dev) {
    return spl_spmv_ex(ctx, a, x_dev, y_dev, SPL_SPMV_AUTO);
}

int spl_spmv_host(spl_ctx *ctx, const spl_mat *a, const void *x_host, void *y_host) {
    API_BEGIN(ctx)
    MatUse use_a(ctx, a);
    SPL_REQUIRE(a && x_host && y_host, SPL_ERR_ARG, "NULL argument");
    const size_t vs = a->vsize();
    Tmp<unsigned char> x(ctx, (size_t)a->ncols * vs), y(ctx, (size_t)a->nrows * vs);
    if (a->wide() || !spmv_host_pipelined(ctx, a, x_host, y_host, x, y)) {
        SPL_CUDA(cudaMemcpyAsync(x, x_host, (size_t)a->ncols * vs, cudaMemcpyHostToDevice, ctx->stream));
        if (a->wide()) wide_spmv(ctx, a, x, y);
        else spmv(ctx, a, x, y, SPL_SPMV_AUTO, 0);
        SPL_CUDA(cudaMemcpyAsync(y_host, y, (size_t)a->nrows * vs, cudaMemcpyDeviceToHost, ctx->stream));
    }
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    API_END(ctx)
}

int spl_spmv_choice(spl_ctx *ctx, const spl_mat *a, int *kernel, int *lanes_per_row) {
    API_BEGIN(ctx)
    SPL_REQUIRE(a, SPL_ERR_ARG, "NULL handle");
    if (a->wide()) {                      // 64-bit positions: the vector kernel, lanes from the mean row length
        if (kernel) *kernel = SPL_SPMV_VECTOR;
        if (lanes_per_row) *lanes_per_row = 0;
        return SPL_OK;
    }
    a = csr_form(ctx, a);                 // a CSC matrix is planned on its CSR form
    spmv_plan(ctx, const_cast<spl_mat *>(a));
    if (kernel) *kernel = a->plan_kernel;
    if (lanes_per_row) *lanes_per_row = a->plan_lanes;
    API_END(ctx)
}

int spl_mat_info(const spl_mat *m, int *format, int *dtype, uint64_t *nrows, uint64_t *ncols,
                 uint64_t *nnz) {
    if (!m) return SPL_ERR_ARG;
    if (format) *format = m->format;
    if (dtype) *dtype = m->dtype;
    if (nrows) *nrows = m->nrows;
    if (ncols) *ncols = m->ncols;
    if (nnz) *nnz = m->entries();
    return SPL_OK;
}

int spl_mat_download(spl_ctx *ctx, const spl_mat *m, uint64_t *ptr, uint64_t *ind, void *val) {
    API_BEGIN(ctx)
    MatUse use_m(ctx, m);
    SPL_REQUIRE(m, SPL_ERR_ARG, "NULL handle");
    const size_t np = (size_t)m->nmajor() + 1;
    if (m->wide()) {                      // pointers are already uint64; indices widen in chunks
        if (ptr) SPL_CUDA(cudaMemcpyAsync(ptr, m->ptr64, np * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (ind) {
            constexpr uint64_t kChunk = 1ull << 26;
            Tmp<uint64_t> stage(ctx, kChunk);
            for (uint64_t at = 0; at < m->nnz64; at += kChunk) {
                const uint64_t cnt = std::min(kChunk, m->nnz64 - at);
                widen_u32(ctx, m->ind + at, stage, cnt);
                SPL_CUDA(cudaMemcpyAsync(ind + at, stage, cnt * 8, cudaMemcpyDeviceToHost, ctx->stream));
            }
        }
        if (val) SPL_CUDA(cudaMemcpyAsync(val, m->val, (size_t)m->nnz64 * m->vsize(), cudaMemcpyDeviceToHost, ctx->stream));
        SPL_CUDA(cudaStreamSynchronize(ctx->stream));
        return SPL_OK;
    }
    Tmp<uint64_t> wide(ctx, np > m->nnz ? np : m->nnz);
    if (ptr) {
        widen_u32(ctx, m->ptr, wide, np);
        SPL_CUDA(cudaMemcpyAsync(ptr, wide, np * 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (ind && m->nnz) {
        widen_u32(ctx, m->ind, wide, m->nnz);
        SPL_CUDA(cudaMemcpyAsync(ind, wide, (size_t)m->nnz * 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (val && m->nnz)
        SPL_CUDA(cudaMemcpyAsync(val, m->val, (size_t)m->nnz * m->vsize(), cudaMemcpyDeviceToHost,
                                 ctx->stream));
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    API_END(ctx)
}

int spl_mat_set_values(spl_ctx *ctx, spl_mat *m, const void *val) {
    API_BEGIN(ctx)
    require_narrow(m, "spl_mat_set_values");
    MatUse use_m(ctx, m);
    SPL_REQUIRE(m && (val || m->nnz == 0), SPL_ERR_ARG, "NULL argument");
    if (m->nnz) {
        SPL_CUDA(cudaMemcpyAsync(m->val, val, (size_t)m->nnz * m->vsize(), cudaMemcpyHostToDevice, ctx->stream));
        SPL_CUDA(cudaStreamSynchronize(ctx->stream));      // the caller may reuse its buffer at once
        drop_value_copies(ctx, m);                         // copies of the old values: CSR twin, sliced SpMV copy, band value codes
    }
    API_END(ctx)
}

int spl_mat_device_ptrs(const spl_mat *m, const uint32_t **ptr_dev, const uint32_t **ind_dev,
                        const void **val_dev) {
    if (!m) return SPL_ERR_ARG;
    if (ptr_dev) *ptr_dev = m->ptr;
    if (ind_dev) *ind_dev = m->ind;
    if (val_dev) *val_dev = m->val;
    return SPL_OK;
}

int spl_mat_device_ptr64(const spl_mat *m, const uint64_t **ptr64_dev) {
    if (!m || !ptr64_dev) return SPL_ERR_ARG;
    *ptr64_dev = m->ptr64;
    return SPL_OK;
}

int spl_mat_to_coo(spl_ctx *ctx, const spl_mat *m, uint64_t *row, uint64_t *col, void *val) {
    API_BEGIN(ctx)
    require_narrow(m, "spl_mat_to_coo");
    MatUse use_m(ctx, m);
    SPL_REQUIRE(m, SPL_ERR_ARG, "NULL handle");
    if (m->nnz) {
        SPL_REQUIRE(row && col && val, SPL_ERR_ARG, "NULL array");
        Tmp<uint32_t> major(ctx, m->nnz);
        Tmp<uint64_t> wide(ctx, m->nnz);
        expand_major(ctx, m->nmajor(), m->nnz, m->ptr, major);
        uint64_t *major_out = m->format == SPL_CSR ? row : col;
        uint64_t *minor_out = m->format == SPL_CSR ? col : row;
        widen_u32(ctx, major, wide, m->nnz);
        SPL_CUDA(cudaMemcpyAsync(major_out, wide, (size_t)m->nnz * 8, cudaMemcpyDeviceToHost,
                                 ctx->stream));
        widen_u32(ctx, m->ind, wide, m->nnz);
        SPL_CUDA(cudaMemcpyAsync(minor_out, wide, (size_t)m->nnz * 8, cudaMemcpyDeviceToHost,
                                 ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(val, m->val, (size_t)m->nnz * m->vsize(), cudaMemcpyDeviceToHost,
                                 ctx->stream));
        SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    API_END(ctx)
}

int spl_mat_to_coo_dev(spl_ctx *ctx, const spl_mat *m, uint32_t *row_dev, uint32_t *col_dev, void *val_dev) {
    API_BEGIN(ctx)
    require_narrow(m, "spl_mat_to_coo_dev");
    MatUse use_m(ctx, m);
    SPL_REQUIRE(m, SPL_ERR_ARG, "NULL handle");
    if (m->nnz) {
        SPL_REQUIRE(row_dev && col_dev && val_dev, SPL_ERR_ARG, "NULL array");
        expand_major(ctx, m->nmajor(), m->nnz, m->ptr, m->format == SPL_CSR ? row_dev : col_dev);
        SPL_CUDA(cudaMemcpyAsync(m->format == SPL_CSR ? col_dev : row_dev, m->ind, (size_t)m->nnz * 4,
                                 cudaMemcpyDeviceToDevice, ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(val_dev, m->val, (size_t)m->nnz * m->vsize(), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    API_END(ctx)
}

int spl_mat_read_entries(spl_ctx *ctx, const spl_mat *m, uint64_t start, uint64_t count, uint64_t *row,
                         uint64_t *col, void *val) {
    API_BEGIN(ctx)
    MatUse use_m(ctx, m);
    SPL_REQUIRE(m, SPL_ERR_ARG, "NULL handle");
    SPL_REQUIRE(start <= m->entries() && count <= m->entries() - start, SPL_ERR_ARG, "entry range outside the matrix");
    SPL_REQUIRE(count < kMaxEntries, SPL_ERR_ARG, "one chunk holds fewer than 2^32 - 65536 entries");
    if (count) {
        SPL_REQUIRE(row && col && val, SPL_ERR_ARG, "NULL array");
        Tmp<uint64_t> major(ctx, count), minor(ctx, count);
        if (m->wide()) wide_entry_range(ctx, m, start, (uint32_t)count, major, minor);
        else entry_range(ctx, m, (uint32_t)start, (uint32_t)count, major, minor);
        SPL_CUDA(cudaMemcpyAsync(m->format == SPL_CSR ? row : col, major, count * 8, cudaMemcpyDeviceToHost, ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(m->format == SPL_CSR ? col : row, minor, count * 8, cudaMemcpyDeviceToHost, ctx->stream));
        SPL_CUDA(cudaMemcpyAsync(val, static_cast<const unsigned char *>(m->val) + start * m->vsize(), count * m->vsize(),
                                 cudaMemcpyDeviceToHost, ctx->stream));
        SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    API_END(ctx)
}

int spl_mat_free(spl_ctx *ctx, spl_mat *m) {
    API_BEGIN(ctx)
    free_mat(ctx, m);
    API_END(ctx)
}

// ---- row sharding across GPUs (SURVEY.md 8e) ------------------------------------------------

int spl_coo_route_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                      uint64_t len, const uint32_t *row_dev, const uint32_t *col_dev,
                      const void *val_dev, int world, const uint64_t *major_starts,
                      uint64_t *keys_out_dev, void *vals_out_dev, uint64_t *counts_host) {
    API_BEGIN(ctx)
    check_enums(format, dtype);
    check_dims(ctx, nrows, ncols);
    SPL_REQUIRE(len < kMaxEntries, SPL_ERR_UNSUPPORTED, "COO length must be below 2^32 - 65536");
    SPL_REQUIRE(major_starts && counts_host, SPL_ERR_ARG, "NULL argument");
    SPL_REQUIRE(len == 0 || (row_dev && col_dev && val_dev && keys_out_dev && vals_out_dev),
                SPL_ERR_ARG, "NULL COO array");
    route_coo_dev(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, (uint32_t)len, row_dev, col_dev,
                  val_dev, world, major_starts, keys_out_dev, vals_out_dev, counts_host);
    API_END(ctx)
}

int spl_coo_route_count_dev(spl_ctx *ctx, int format, uint64_t nrows, uint64_t ncols, uint64_t len,
                            const uint32_t *row_dev, const uint32_t *col_dev, int world,
                            const uint64_t *major_starts, uint64_t *counts_host) {
    API_BEGIN(ctx)
    check_enums(format, SPL_F64);
    check_dims(ctx, nrows, ncols);
    SPL_REQUIRE(len < kMaxEntries, SPL_ERR_UNSUPPORTED, "COO length must be below 2^32 - 65536");
    SPL_REQUIRE(major_starts && counts_host && (len == 0 || (row_dev && col_dev)), SPL_ERR_ARG, "NULL argument");
    route_count_dev(ctx, format, (uint32_t)nrows, (uint32_t)ncols, (uint32_t)len, row_dev, col_dev, world,
                    major_starts, counts_host);
    API_END(ctx)
}

int spl_coo_route_peers_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                            uint64_t len, const uint32_t *row_dev, const uint32_t *col_dev,
                            const void *val_dev, int world, const uint64_t *major_starts,
                            void *const *key_bufs, void *const *val_bufs, const uint64_t *dst_offsets) {
    API_BEGIN(ctx)
    check_enums(format, dtype);
    check_dims(ctx, nrows, ncols);
    SPL_REQUIRE(len < kMaxEntries, SPL_ERR_UNSUPPORTED, "COO length must be below 2^32 - 65536");
    SPL_REQUIRE(major_starts && key_bufs && val_bufs && dst_offsets, SPL_ERR_ARG, "NULL argument");
    SPL_REQUIRE(len == 0 || (row_dev && col_dev && val_dev), SPL_ERR_ARG, "NULL COO array");
    route_coo_peers_dev(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, (uint32_t)len, row_dev, col_dev,
                        val_dev, world, major_starts, key_bufs, val_bufs, dst_offsets);
    API_END(ctx)
}

int spl_mat_from_packed_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                            uint64_t len, const uint64_t *keys_dev, const void *vals_dev, int dedup,
                            int dropzero, spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(out, SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    check_enums(format, dtype);
    check_dims(ctx, nrows, ncols);
    SPL_REQUIRE(len < kMaxEntries, SPL_ERR_UNSUPPORTED, "COO length must be below 2^32 - 65536");
    SPL_REQUIRE(len == 0 || (keys_dev && vals_dev), SPL_ERR_ARG, "NULL COO array");
    *out = assemble_from_packed_dev(ctx, format, dtype, (uint32_t)nrows, (uint32_t)ncols, (uint32_t)len,
                                    keys_dev, vals_dev, dedup, dropzero);
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_peer_alloc(spl_ctx *ctx, uint64_t bytes, void **dev_ptr, unsigned char *handle_out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(dev_ptr && handle_out, SPL_ERR_ARG, "NULL argument");
    *dev_ptr = nullptr;
    void *p = nullptr;
    SPL_CUDA(cudaMalloc(&p, bytes ? bytes : 1));        // plain cudaMalloc: IPC-exportable
    cudaIpcMemHandle_t h;
    static_assert(sizeof(h) == SPL_IPC_HANDLE_BYTES, "CUDA IPC handle size");
    cudaError_t e = cudaMemset(p, 0, bytes ? bytes : 1);
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        throw Error{SPL_ERR_CUDA, std::string("spl_peer_alloc: ") + cudaGetErrorString(e)};
    }
    std::memcpy(handle_out, &h, sizeof(h));
    *dev_ptr = p;
    API_END(ctx)
}

int spl_peer_open(spl_ctx *ctx, const unsigned char *handle, void **peer_ptr) {
    API_BEGIN(ctx)
    SPL_REQUIRE(handle && peer_ptr, SPL_ERR_ARG, "NULL argument");
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    SPL_CUDA(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    API_END(ctx)
}

int spl_peer_close(spl_ctx *ctx, void *peer_ptr) {
    API_BEGIN(ctx)
    if (peer_ptr) {
        SPL_CUDA(cudaStreamSynchronize(ctx->stream));
        SPL_CUDA(cudaIpcCloseMemHandle(peer_ptr));
    }
    API_END(ctx)
}

int spl_peer_free(spl_ctx *ctx, void *dev_ptr) {
    API_BEGIN(ctx)
    if (dev_ptr) {
        SPL_CUDA(cudaStreamSynchronize(ctx->stream));
        SPL_CUDA(cudaFree(dev_ptr));
    }
    API_END(ctx)
}

int spl_peer_barrier(spl_ctx *ctx, int world, int rank, void *const *flag_ptrs, uint32_t epoch,
                     uint32_t timeout_ms) {
    API_BEGIN(ctx)
    SPL_REQUIRE(flag_ptrs, SPL_ERR_ARG, "NULL argument");
    peer_barrier(ctx, world, rank, flag_ptrs, epoch, timeout_ms);
    API_END(ctx)
}

int spl_peer_barrier_halo(spl_ctx *ctx, int world, int rank, void *const *flag_ptrs, uint32_t epoch,
                          uint32_t timeout_ms, int dtype, const uint64_t *starts, void *const *x_slices,
                          uint64_t halo_left, uint64_t halo_right) {
    API_BEGIN(ctx)
    check_enums(SPL_CSR, dtype);
    SPL_REQUIRE(flag_ptrs && starts && x_slices, SPL_ERR_ARG, "NULL argument");
    SPL_REQUIRE(halo_left < (1ull << 31) && halo_right < (1ull << 31), SPL_ERR_UNSUPPORTED, "halo too wide");
    peer_barrier_halo(ctx, world, rank, flag_ptrs, epoch, timeout_ms, dtype == SPL_F32 ? 4 : 8, starts, x_slices,
                      (uint32_t)halo_left, (uint32_t)halo_right);
    API_END(ctx)
}

int spl_spmv_window(spl_ctx *ctx, const spl_mat *a, const void *x_window_dev, uint64_t window_start,
                    uint64_t window_len, void *y_dev) {
    API_BEGIN(ctx)
    require_narrow(a, "spl_spmv_window");
    MatUse use_a(ctx, a);
    SPL_REQUIRE(a && x_window_dev && y_dev, SPL_ERR_ARG, "NULL argument");
    spmv_window(ctx, a, x_window_dev, window_start, window_len, y_dev);
    API_END(ctx)
}

int spl_spmv_footprint(spl_ctx *ctx, const spl_mat *a, uint64_t *col_min, uint64_t *col_max) {
    API_BEGIN(ctx)
    require_narrow(a, "spl_spmv_footprint");
    MatUse use_a(ctx, a);
    SPL_REQUIRE(a, SPL_ERR_ARG, "NULL handle");
    a = csr_form(ctx, a);
    spmv_plan(ctx, const_cast<spl_mat *>(a));
    if (col_min) *col_min = a->nnz ? a->col_min : 0;
    if (col_max) *col_max = a->nnz ? a->col_max : 0;
    API_END(ctx)
}

int spl_spmv_transpose_window(spl_ctx *ctx, const spl_mat *a, const void *x_dev, void *y_window_dev) {
    API_BEGIN(ctx)
    require_narrow(a, "spl_spmv_transpose_window");
    MatUse use_a(ctx, a);
    SPL_REQUIRE(a && x_dev && y_window_dev, SPL_ERR_ARG, "NULL argument");
    spmv_transpose_window(ctx, a, x_dev, y_window_dev);
    API_END(ctx)
}

int spl_peer_reduce_windows(spl_ctx *ctx, int dtype, int world, int rank, const uint64_t *col_starts,
                            const uint64_t *windows, const void *const *partials, void *const *flag_ptrs, uint32_t epoch,
                            uint32_t timeout_ms, void *y_local_dev) {
    API_BEGIN(ctx)
    check_enums(SPL_CSR, dtype);
    SPL_REQUIRE(col_starts && windows && partials, SPL_ERR_ARG, "NULL argument");
    SPL_REQUIRE(world >= 1 && world <= SPL_MAX_PEERS && rank >= 0 && rank < world, SPL_ERR_ARG,
                "world must be 1..8 and rank inside it");
    SPL_REQUIRE(col_starts[0] == 0, SPL_ERR_ARG, "col_starts must begin at 0");
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(col_starts[g] <= col_starts[g + 1], SPL_ERR_ARG, "col_starts must be non-decreasing");
        SPL_REQUIRE(!flag_ptrs || flag_ptrs[g], SPL_ERR_ARG, "NULL flag block");
    }
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(windows[2 * g] <= windows[2 * g + 1] && windows[2 * g + 1] <= col_starts[world], SPL_ERR_ARG,
                    "a window lies outside the columns [0, col_starts[world])");
        SPL_REQUIRE(partials[g] || windows[2 * g] == windows[2 * g + 1], SPL_ERR_ARG, "NULL partial of a non-empty window");
    }
    SPL_REQUIRE(y_local_dev || col_starts[rank] == col_starts[rank + 1], SPL_ERR_ARG, "NULL y");
    peer_reduce_windows(ctx, dtype, world, rank, col_starts, windows, partials, flag_ptrs, epoch, timeout_ms, y_local_dev);
    API_END(ctx)
}

int spl_peer_pull(spl_ctx *ctx, int dtype, int world, int rank, const uint64_t *starts,
                  const void *const *slices, void *x_full_dev) {
    API_BEGIN(ctx)
    check_enums(SPL_CSR, dtype);
    SPL_REQUIRE(starts && slices && x_full_dev, SPL_ERR_ARG, "NULL argument");
    peer_pull(ctx, world, rank, dtype == SPL_F32 ? 4 : 8, starts, slices, x_full_dev);
    API_END(ctx)
}

int spl_peer_gather_rows(spl_ctx *ctx, int format, int dtype, uint64_t nmajor, uint64_t nminor, int world, int rank,
                         const uint64_t *starts, const uint64_t *shard_nnz, const void *const *ptr_slices,
                         const void *const *ind_slices, const void *const *val_slices, const spl_mat *by,
                         spl_mat **out) {
    API_BEGIN(ctx)
    SPL_REQUIRE(out, SPL_ERR_ARG, "out is NULL");
    *out = nullptr;
    SPL_REQUIRE(by && starts && shard_nnz && ptr_slices && ind_slices && val_slices, SPL_ERR_ARG, "NULL argument");
    check_enums(format, dtype);
    SPL_REQUIRE(world >= 1 && world <= SPL_MAX_PEERS && rank >= 0 && rank < world, SPL_ERR_ARG,
                "world must be 1..8 and rank inside it");
    require_narrow(by, "spl_peer_gather_rows");
    SPL_REQUIRE(by->format == format && by->dtype == dtype, SPL_ERR_ARG,
                "spl_peer_gather_rows: by must have the gathered matrix's format and scalar type");
    SPL_REQUIRE(starts[0] == 0, SPL_ERR_ARG, "starts must begin at 0");
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(starts[g] <= starts[g + 1], SPL_ERR_ARG, "starts must be non-decreasing");
        SPL_REQUIRE(starts[g] == starts[g + 1] || (ptr_slices[g] && ind_slices[g] && val_slices[g]), SPL_ERR_ARG,
                    "NULL slice of a rank that owns majors");
        SPL_REQUIRE(shard_nnz[g] < kMaxEntries, SPL_ERR_UNSUPPORTED, "a shard holds 2^32 - 65536 entries or more");
    }
    SPL_REQUIRE(starts[world] == nmajor && by->nminor() == nmajor, SPL_ERR_SHAPE,
                "spl_peer_gather_rows: starts[world] and by's minor dimension must equal nmajor");
    SPL_REQUIRE(nminor > 0 && nminor < (1ull << 32), SPL_ERR_UNSUPPORTED, "nminor must be in 1 .. 2^32 - 1");
    MatUse use_by(ctx, by);
    *out = peer_gather_rows(ctx, format, dtype, (uint32_t)nmajor, (uint32_t)nminor, world, starts, shard_nnz,
                            ptr_slices, ind_slices, val_slices, by);
    publish_mat(ctx, *out);
    API_END(ctx)
}

int spl_peer_barrier_status(spl_ctx *ctx, int *timed_out) {
    API_BEGIN(ctx)
    uint32_t w = 0;
    read_back(ctx, ctx->d_scratch + 32, &w, 1);
    if (timed_out) *timed_out = (int)w;
    if (w) SPL_CUDA(cudaMemsetAsync(ctx->d_scratch + 32, 0, sizeof(uint32_t), ctx->stream));   // report once
    SPL_REQUIRE(w == 0, SPL_ERR_CUDA, "spl_peer_barrier timed out waiting for a peer");
    API_END(ctx)
}

int spl_spmv_peer(spl_ctx *ctx, const spl_mat *a_local, int world, int rank,
                  const uint64_t *col_starts, const void *const *x_slices, void *y_dev) {
    API_BEGIN(ctx)
    require_narrow(a_local, "spl_spmv_peer");
    MatUse use_a_local(ctx, a_local);
    SPL_REQUIRE(a_local && col_starts && x_slices && y_dev, SPL_ERR_ARG, "NULL argument");
    SPL_REQUIRE(world >= 1 && world <= SPL_MAX_PEERS && rank >= 0 && rank < world, SPL_ERR_ARG,
                "world must be 1..8 and rank inside it");
    SPL_REQUIRE(col_starts[0] == 0 && col_starts[world] == a_local->ncols, SPL_ERR_SHAPE,
                "col_starts must run from 0 to A.ncols()");
    PeerX px{};
    px.world = world;
    px.rank = rank;
    for (int g = 0; g <= SPL_MAX_PEERS; ++g) px.start[g] = (uint32_t)col_starts[g < world ? g : world];
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(col_starts[g] <= col_starts[g + 1], SPL_ERR_ARG, "col_starts must be non-decreasing");
        SPL_REQUIRE(x_slices[g] || col_starts[g] == col_starts[g + 1], SPL_ERR_ARG, "NULL x slice");
        px.slice[g] = x_slices[g];
    }
    spmv_peer(ctx, a_local, px, y_dev);
    API_END(ctx)
}

int spl_spmv_gather_fused(spl_ctx *ctx, int dtype, uint64_t nrows_local, int world, int rank,
                          const uint64_t *col_starts, const void *const *x_slices, int nblocks,
                          const uint32_t *block_first, const uint32_t *block_ptr_dev, uint64_t block_ptr_stride,
                          const uint32_t *tile_entries_max, const uint32_t *block_ind_dev, const void *block_val_dev, void *x_full_dev, void *y_dev,
                          uint32_t *ready_dev, uint32_t epoch, uint64_t nnz_local, void *const *flag_ptrs,
                          uint32_t barrier_epoch, uint32_t timeout_ms, uint64_t *timeline_dev) {
    API_BEGIN(ctx)
    check_enums(SPL_CSR, dtype);
    SPL_REQUIRE(col_starts && x_slices && block_ptr_dev && x_full_dev && y_dev && ready_dev, SPL_ERR_ARG, "NULL argument");
    SPL_REQUIRE(world >= 1 && world <= SPL_MAX_PEERS && rank >= 0 && rank < world, SPL_ERR_ARG,
                "world must be 1..8 and rank inside it");
    SPL_REQUIRE(nrows_local > 0 && nrows_local < (1ull << 32) && col_starts[world] < (1ull << 32), SPL_ERR_UNSUPPORTED,
                "dimensions must be below 2^32");
    SPL_REQUIRE(epoch > 0, SPL_ERR_ARG, "epoch counts from 1 and grows by one per call");
    SPL_REQUIRE(tile_entries_max, SPL_ERR_ARG, "NULL tile_entries_max");
    SPL_REQUIRE(block_ptr_stride % 4 == 0 && block_ptr_stride > nrows_local && block_ptr_stride < (1ull << 32), SPL_ERR_ARG,
                "block_ptr_stride must be a multiple of 4 above nrows_local");
    SPL_REQUIRE(((uintptr_t)block_ptr_dev | (uintptr_t)block_ind_dev | (uintptr_t)block_val_dev) % 16 == 0, SPL_ERR_ARG,
                "the block arrays must be 16-byte aligned");
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(col_starts[g] <= col_starts[g + 1], SPL_ERR_ARG, "col_starts must be non-decreasing");
        SPL_REQUIRE(x_slices[g] || col_starts[g] == col_starts[g + 1], SPL_ERR_ARG, "NULL x slice");
    }
    spmv_gather_fused(ctx, dtype, (uint32_t)nrows_local, world, rank, col_starts, x_slices, nblocks, block_first,
                      block_ptr_dev, (uint32_t)block_ptr_stride, tile_entries_max, block_ind_dev, block_val_dev, x_full_dev, y_dev, ready_dev, epoch,
                      (double)nnz_local / (double)nrows_local, flag_ptrs, barrier_epoch, timeout_ms,
                      reinterpret_cast<unsigned long long *>(timeline_dev));
    API_END(ctx)
}

int spl_spmv_peer_host(spl_ctx *ctx, const spl_mat *a_local, int world, int rank, const uint64_t *col_starts,
                       void *const *x_slices, void *const *flag_ptrs, uint32_t epoch, uint32_t timeout_ms,
                       const void *x_host_local, void *y_host_local) {
    API_BEGIN(ctx)
    require_narrow(a_local, "spl_spmv_peer_host");
    MatUse use_a_local(ctx, a_local);
    SPL_REQUIRE(a_local && col_starts && x_slices && flag_ptrs && y_host_local, SPL_ERR_ARG, "NULL argument");
    SPL_REQUIRE(world >= 1 && world <= SPL_MAX_PEERS && rank >= 0 && rank < world, SPL_ERR_ARG,
                "world must be 1..8 and rank inside it");
    SPL_REQUIRE(col_starts[0] == 0 && col_starts[world] == a_local->ncols, SPL_ERR_SHAPE,
                "col_starts must run from 0 to A.ncols()");
    PeerX px{};
    px.world = world;
    px.rank = rank;
    for (int g = 0; g <= SPL_MAX_PEERS; ++g) px.start[g] = (uint32_t)col_starts[g < world ? g : world];
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(col_starts[g] <= col_starts[g + 1], SPL_ERR_ARG, "col_starts must be non-decreasing");
        SPL_REQUIRE(x_slices[g] || col_starts[g] == col_starts[g + 1], SPL_ERR_ARG, "NULL x slice");
        px.slice[g] = x_slices[g];
    }
    SPL_REQUIRE(x_host_local || col_starts[rank] == col_starts[rank + 1], SPL_ERR_ARG, "NULL x");
    Tmp<unsigned char> y(ctx, (size_t)a_local->nrows * a_local->vsize());
    spmv_peer_host(ctx, a_local, px, flag_ptrs, epoch, timeout_ms, x_host_local, y_host_local, y);
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    uint32_t failed = 0;
    read_back(ctx, ctx->d_scratch + 32, &failed, 1);
    if (failed) SPL_CUDA(cudaMemsetAsync(ctx->d_scratch + 32, 0, sizeof(uint32_t), ctx->stream));
    SPL_REQUIRE(failed == 0, SPL_ERR_CUDA, "spl_spmv_peer_host: the barrier timed out waiting for a peer (y holds NaN)");
    API_END(ctx)
}

}  // extern "C"
#pragma GCC visibility pop
