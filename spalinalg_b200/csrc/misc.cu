// misc.cu — streaming helpers around the hot path: negate (src/csr/ops/neg.rs:5-18),
// CsrMatrix::new validation (src/csr.rs:144-156), index narrowing/widening between the host's
// usize and the device's uint32, eye (src/csr.rs:179-188), rowptr expansion (src/csr.rs:303-316).
#include "kernels.cuh"

namespace spl {

namespace {

template <typename T>
__global__ void negate_kernel(const T *__restrict__ in, T *__restrict__ out, uint32_t n) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = flip_sign(in[i]);   // 0.0 -> -0.0, NaN payload kept
}

// assertion 7: ptr non-decreasing (src/csr.rs:150)
__global__ void validate_ptr_kernel(const uint32_t *__restrict__ ptr, uint32_t nmajor,
                                    uint32_t *fail) {
    const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m < nmajor && ptr[m] > ptr[m + 1]) atomicMin(fail, 7u);
}

// assertion 8: index in range (:151); assertion 9: strictly increasing in a segment (:152-156).
// Streaming formulation without any search: count the descents ind[p] >= ind[p+1] over all
// neighbouring entries (D) and the descents that sit exactly on the start of a non-empty
// segment (R); every R is also a D, so the segments are strictly increasing iff D == R.
__global__ void validate_ind_kernel(const uint32_t *__restrict__ ptr,
                                    const uint32_t *__restrict__ ind, uint32_t nmajor,
                                    uint32_t nminor, uint32_t nnz, uint32_t *fail,
                                    unsigned long long *counters) {
    unsigned long long d = 0, r = 0;
    bool oob = false;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (uint64_t p = tid; p < nnz; p += stride) {
        const uint32_t c = ind[p];
        oob |= c >= nminor;
        if (p + 1 < nnz && ind[p + 1] <= c) ++d;
    }
    for (uint64_t m = tid; m < nmajor; m += stride) {
        const uint32_t q = ptr[m];
        if (q > 0 && q < nnz && ptr[m + 1] > q && ind[q] <= ind[q - 1]) ++r;
    }
    if (__any_sync(0xffffffffu, oob) && lane_id() == 0) atomicMin(fail, 8u);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        d += __shfl_xor_sync(0xffffffffu, d, o);
        r += __shfl_xor_sync(0xffffffffu, r, o);
    }
    if (lane_id() == 0) {
        if (d) atomicAdd(counters, d);
        if (r) atomicAdd(counters + 1, r);
    }
}

__global__ void narrow_kernel(const uint64_t *__restrict__ src, uint32_t *__restrict__ dst, size_t n,
                              uint64_t limit, uint32_t *flag) {
    uint32_t bad = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (size_t)gridDim.x * blockDim.x) {
        const uint64_t v = src[i];
        bad |= v >= limit;
        dst[i] = v > 0xffffffffull ? 0xffffffffu : (uint32_t)v;
    }
    if (__any_sync(0xffffffffu, bad) && lane_id() == 0) atomicOr(flag, 1u);
}

__global__ void widen_kernel(const uint32_t *__restrict__ src, uint64_t *__restrict__ dst, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

template <typename T>
__global__ void eye_kernel(uint32_t size, uint32_t *ptr, uint32_t *ind, T *val) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= size) ptr[i] = (uint32_t)i;
    if (i < size) {
        ind[i] = (uint32_t)i;
        val[i] = (T)1;
    }
}

// LPR lanes per segment write the segment's index over its entries: consecutive lanes, consecutive
// entries, so the stores coalesce (a search per entry was measured 6x slower).
template <int LPR>
__global__ void __launch_bounds__(256)
expand_major_kernel(const uint32_t *__restrict__ ptr, uint32_t nmajor, uint32_t *__restrict__ out) {
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t m = gtid / LPR;
    if (m >= nmajor) return;
    const uint32_t e = __ldg(ptr + m + 1);
    for (uint32_t p = __ldg(ptr + m) + (uint32_t)(gtid % LPR); p < e; p += LPR) out[p] = (uint32_t)m;
}

// major index and widened minor index of the stored entries [start, start + count): one search of the
// pointer array per entry (chunks of an iterator are small; the whole-matrix form uses expand_major)
__global__ void __launch_bounds__(256)
entry_range_kernel(const uint32_t *__restrict__ ptr, const uint32_t *__restrict__ ind, uint32_t nmajor, uint32_t start,
                   uint32_t count, uint64_t *__restrict__ major_out, uint64_t *__restrict__ minor_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint32_t p = start + i;
    major_out[i] = upper_bound_u32(ptr, 0u, nmajor + 1u, p) - 1u;      // ptr[m] <= p < ptr[m + 1]
    minor_out[i] = ind[p];
}

inline unsigned stream_grid(spl_ctx *ctx, size_t n) {
    unsigned g = div_up(n ? n : 1, 256 * 4);
    unsigned cap = (unsigned)ctx->num_sms * 16u;
    return g < cap ? (g ? g : 1) : cap;
}

}  // namespace

void negate(spl_ctx *ctx, int dtype, uint32_t nnz, const void *val, void *out) {
    if (nnz == 0) return;
    if (dtype == SPL_F32)
        negate_kernel<float><<<stream_grid(ctx, nnz), 256, 0, ctx->stream>>>((const float *)val,
                                                                            (float *)out, nnz);
    else
        negate_kernel<double><<<stream_grid(ctx, nnz), 256, 0, ctx->stream>>>((const double *)val,
                                                                             (double *)out, nnz);
    check_launch(ctx, "negate");
}

int validate_compressed(spl_ctx *ctx, uint32_t nmajor, uint32_t nminor, uint32_t nnz,
                        const uint32_t *ptr, const uint32_t *ind) {
    uint32_t fail = 0xffffffffu;
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0xff, sizeof(uint32_t), ctx->stream));
    validate_ptr_kernel<<<div_up(nmajor, 256), 256, 0, ctx->stream>>>(ptr, nmajor, ctx->d_scratch);
    check_launch(ctx, "validate_ptr");
    read_back(ctx, ctx->d_scratch, &fail, 1);
    if (fail != 0xffffffffu) return (int)fail;
    if (nnz == 0) return 0;
    // ptr is monotone with ptr[0]==0, ptr[n]==nnz (checked by the caller): every segment is inside ind
    unsigned long long *counters = reinterpret_cast<unsigned long long *>(ctx->d_scratch + 2);
    SPL_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned long long), ctx->stream));
    validate_ind_kernel<<<stream_grid(ctx, nnz), 256, 0, ctx->stream>>>(ptr, ind, nmajor, nminor, nnz,
                                                                       ctx->d_scratch, counters);
    check_launch(ctx, "validate_ind");
    uint32_t w[6];
    read_back(ctx, ctx->d_scratch, w, 6);
    if (w[0] != 0xffffffffu) return (int)w[0];
    const bool increasing = w[2] == w[4] && w[3] == w[5];   // D == R
    return increasing ? 0 : 9;
}

void narrow_u64(spl_ctx *ctx, const uint64_t *src, uint32_t *dst, size_t n, uint64_t limit,
                uint32_t *d_flag) {
    if (n == 0) return;
    narrow_kernel<<<stream_grid(ctx, n), 256, 0, ctx->stream>>>(src, dst, n, limit, d_flag);
    check_launch(ctx, "narrow");
}

void widen_u32(spl_ctx *ctx, const uint32_t *src, uint64_t *dst, size_t n) {
    if (n == 0) return;
    widen_kernel<<<stream_grid(ctx, n), 256, 0, ctx->stream>>>(src, dst, n);
    check_launch(ctx, "widen");
}

void fill_eye(spl_ctx *ctx, int dtype, uint32_t size, uint32_t *ptr, uint32_t *ind, void *val) {
    const unsigned grid = div_up((uint64_t)size + 1, 256);
    if (dtype == SPL_F32) eye_kernel<float><<<grid, 256, 0, ctx->stream>>>(size, ptr, ind, (float *)val);
    else eye_kernel<double><<<grid, 256, 0, ctx->stream>>>(size, ptr, ind, (double *)val);
    check_launch(ctx, "eye");
}

void expand_major(spl_ctx *ctx, uint32_t nmajor, uint32_t nnz, const uint32_t *ptr, uint32_t *out) {
    if (nnz == 0) return;
    const double mean = (double)nnz / nmajor;
    if (mean <= 2.0)
        expand_major_kernel<1><<<div_up(nmajor, 256), 256, 0, ctx->stream>>>(ptr, nmajor, out);
    else if (mean <= 12.0)
        expand_major_kernel<4><<<div_up((uint64_t)nmajor * 4, 256), 256, 0, ctx->stream>>>(ptr, nmajor, out);
    else if (mean <= 64.0)
        expand_major_kernel<8><<<div_up((uint64_t)nmajor * 8, 256), 256, 0, ctx->stream>>>(ptr, nmajor, out);
    else
        expand_major_kernel<32><<<div_up((uint64_t)nmajor * 32, 256), 256, 0, ctx->stream>>>(ptr, nmajor, out);
    check_launch(ctx, "expand_major");
}

void entry_range(spl_ctx *ctx, const spl_mat *m, uint32_t start, uint32_t count, uint64_t *major_out,
                 uint64_t *minor_out) {
    if (count == 0) return;
    entry_range_kernel<<<div_up(count, 256), 256, 0, ctx->stream>>>(m->ptr, m->ind, m->nmajor(), start, count, major_out,
                                                                   minor_out);
    check_launch(ctx, "entry_range");
}

spl_mat *new_mat(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols, uint32_t nnz) {
    spl_mat *m = new spl_mat();
    m->format = format;
    m->dtype = dtype;
    m->nrows = nrows;
    m->ncols = ncols;
    m->nnz = nnz;
    try {
        // +4 pointers of slack: the stream SpMV fetches pointer slices in whole 16-byte units
        m->ptr = dalloc<uint32_t>(ctx, (size_t)m->nmajor() + 1 + 4);
        // +16 entries of slack: the SpMV kernels read aligned groups of four entries
        m->ind = dalloc<uint32_t>(ctx, (size_t)nnz + 16);
        m->val = dalloc_bytes(ctx, ((size_t)nnz + 16) * m->vsize());
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    return m;
}

void free_mat(spl_ctx *ctx, spl_mat *m) {
    if (!m) return;
    // readers on other streams first: the blocks go back to the pool in this context's stream order
    if (m->ready && m->home != ctx->stream) {
        // freed by a context other than its creator: the creator's stream may still hold queued readers
        // this context cannot name; rare, so settle it the blunt way
        cudaDeviceSynchronize();
    } else {
        std::lock_guard<std::mutex> lock(m->use_mu);
        for (auto &f : m->foreign) cudaStreamWaitEvent(ctx->stream, f.done, 0);
    }
    for (auto &f : m->foreign) cudaEventDestroy(f.done);
    m->foreign.clear();
    if (m->ready) cudaEventDestroy(m->ready);
    m->ready = nullptr;
    free_mat(ctx, m->twin.exchange(nullptr));
    dfree(ctx, m->ptr);
    dfree(ctx, m->ptr64);
    dfree(ctx, m->ind);
    dfree(ctx, m->val);
    dfree(ctx, m->merge_rows);
    dfree(ctx, m->split_rows);
    dfree(ctx, m->ind_rank);
    dfree(ctx, m->col_order);
    dfree(ctx, m->slice_ptr);
    dfree(ctx, m->slice_ind);
    dfree(ctx, m->slice_val);
    dfree(ctx, m->stream_xhi);
    dfree(ctx, m->stream_cta_rows);
    dfree(ctx, m->stream_xlo0);
    dfree(ctx, m->stream_tile_lo);
    dfree(ctx, m->stream_tile_reg);
    delete m;
}

}  // namespace spl
