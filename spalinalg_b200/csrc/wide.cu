// wide.cu — matrices with 2^32 - 65536 or more stored entries ("wide": 64-bit positions).
//
// The reference indexes everything with usize (src/csr.rs:66-72); the device kernels use 32-bit
// positions because every BASELINE configuration fits them and they halve the pointer traffic.  A
// matrix beyond that (a 2^32-entry f32 matrix is 34 GB: it fits this GPU) keeps a uint64 pointer array
// (`spl_mat::ptr64`; indices stay 32-bit, dimensions stay below 2^32) and is served by the kernels
// below: validation (CsrMatrix::new, src/csr.rs:144-156), SpMV (the vector kernel with 64-bit
// positions), transpose / CSR<->CSC (src/csr.rs:358-406, src/csc/conv/csr.rs:3-53: histogram +
// 64-bit exclusive scan + scatter + per-segment repair, the reference's own three steps),
// download and the chunks of iter().  COO assembly of such a matrix (2^32 - 65536 triplets or more)
// runs in wide_assemble.cu on the scan below.  Everything else on the path (add/sub, mul) answers
// SPL_ERR_UNSUPPORTED for a wide operand.
#include <algorithm>

#include "kernels.cuh"

namespace spl {

namespace {

constexpr uint32_t kWideRepairMax = 256;      // longest output segment the transpose's repair pass ranks

// ---- validation (assertions 7, 8, 9 of CsrMatrix::new) ---------------------------------------
__global__ void wide_validate_ptr_kernel(const uint64_t *__restrict__ ptr, uint32_t nmajor, uint32_t *fail) {
    const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m < nmajor && ptr[m] > ptr[m + 1]) atomicMin(fail, 7u);
}

// same streaming formulation as validate_ind_kernel (misc.cu): descents over all neighbours (D) against
// descents that sit on the start of a non-empty segment (R); strictly increasing segments iff D == R
__global__ void wide_validate_ind_kernel(const uint64_t *__restrict__ ptr, const uint32_t *__restrict__ ind,
                                         uint32_t nmajor, uint32_t nminor, uint64_t nnz, uint32_t *fail,
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
        const uint64_t q = ptr[m];
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

// ---- SpMV: the vector kernel (spmv.cu) with 64-bit positions ---------------------------------
template <typename T, int LPR>
__global__ void __launch_bounds__(256)
wide_spmv_vector_kernel(uint32_t nrows, const uint64_t *__restrict__ ptr, const uint32_t *__restrict__ ind,
                        const T *__restrict__ val, const T *__restrict__ x, T *__restrict__ y) {
    constexpr int U = 4;
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t row = gtid / LPR;
    const uint32_t sub = (uint32_t)(gtid % LPR);
    T acc = (T)0;
    if (row < nrows) {
        uint64_t p = __ldg(ptr + row) + sub;
        const uint64_t e = __ldg(ptr + row + 1);
        for (; p < e; p += U * LPR) {
            uint32_t c[U];
            T v[U], xv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint64_t pu = p + (uint64_t)u * LPR;
                const uint64_t idx = pu < e ? pu : p;
                c[u] = __ldg(ind + idx);
                v[u] = __ldg(val + idx);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) xv[u] = __ldg(x + c[u]);
#pragma unroll
            for (int u = 0; u < U; ++u) acc += p + (uint64_t)u * LPR < e ? v[u] * xv[u] : (T)0;
        }
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (sub == 0 && row < nrows) y[row] = acc;
}

template <typename T, int LPR>
void launch_wide_vector(spl_ctx *ctx, const spl_mat *a, const T *x, T *y) {
    const uint64_t threads = (uint64_t)a->nrows * LPR;
    wide_spmv_vector_kernel<T, LPR><<<div_up(threads, 256), 256, 0, ctx->stream>>>(
        a->nrows, a->ptr64, a->ind, static_cast<const T *>(a->val), x, y);
    check_launch(ctx, "wide_spmv_vector");
}

template <typename T>
void wide_spmv_t(spl_ctx *ctx, const spl_mat *a, const T *x, T *y) {
    const double mean = a->nrows ? (double)a->nnz64 / a->nrows : 0.0;
    int lanes = 1;
    if (mean > 12.0) lanes = 4;
    while (lanes < 32 && lanes * 10 < mean) lanes *= 2;
    switch (lanes) {
        case 1: launch_wide_vector<T, 1>(ctx, a, x, y); break;
        case 2: launch_wide_vector<T, 2>(ctx, a, x, y); break;
        case 4: launch_wide_vector<T, 4>(ctx, a, x, y); break;
        case 8: launch_wide_vector<T, 8>(ctx, a, x, y); break;
        case 16: launch_wide_vector<T, 16>(ctx, a, x, y); break;
        default: launch_wide_vector<T, 32>(ctx, a, x, y); break;
    }
}

// ---- transpose / CSR <-> CSC: histogram, 64-bit exclusive scan, scatter, repair ----------------
__global__ void wide_minor_count_kernel(const uint32_t *__restrict__ ind, uint64_t nnz, uint32_t *__restrict__ counts) {
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (uint64_t)gridDim.x * blockDim.x)
        atomicAdd(counts + ind[p], 1u);
}

__global__ void wide_max_kernel(const uint32_t *__restrict__ a, uint32_t n, uint32_t *__restrict__ out) {
    uint32_t m = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        m = max(m, a[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane_id() == 0 && m) atomicMax(out, m);
}

// Exclusive scan of uint32 counts into uint64 pointers, three kernels: per-tile sums, one-block scan of the
// sums, per-tile downsweep.  n + 1 outputs.
constexpr int WS_THREADS = 256, WS_IPT = 16, WS_TILE = WS_THREADS * WS_IPT;

__device__ __forceinline__ unsigned long long wide_block_scan(unsigned long long v, unsigned long long *ws,
                                                              unsigned long long *total) {
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    unsigned long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += t;
    }
    if (lane == 31) ws[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long s = lane < nwarps ? ws[lane] : 0ull, si = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, si, o);
            if (lane >= (unsigned)o) si += t;
        }
        if (lane < nwarps) ws[lane] = si - s;
        if (lane == 31) ws[nwarps] = si;
    }
    __syncthreads();
    if (total) *total = ws[nwarps];
    return ws[warp] + incl - v;
}

__global__ void __launch_bounds__(WS_THREADS)
wide_scan_reduce_kernel(const uint32_t *__restrict__ in, uint32_t n, unsigned long long *__restrict__ tile_sums) {
    __shared__ unsigned long long ws[WS_THREADS / 32 + 1];
    const uint64_t base = (uint64_t)blockIdx.x * WS_TILE + (uint64_t)threadIdx.x * WS_IPT;
    unsigned long long s = 0;
    for (int i = 0; i < WS_IPT; ++i)
        if (base + i < n) s += in[base + i];
    unsigned long long total;
    wide_block_scan(s, ws, &total);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) wide_scan_spine_kernel(unsigned long long *data, uint32_t m) {
    __shared__ unsigned long long ws[33];
    const uint32_t per = (m + blockDim.x - 1) / blockDim.x;
    const uint64_t lo = (uint64_t)threadIdx.x * per, hi = lo + per < m ? lo + per : m;
    unsigned long long s = 0;
    for (uint64_t i = lo; i < hi; ++i) s += data[i];
    unsigned long long run = wide_block_scan(s, ws, nullptr);
    for (uint64_t i = lo; i < hi; ++i) {
        const unsigned long long v = data[i];
        data[i] = run;
        run += v;
    }
}

__global__ void __launch_bounds__(WS_THREADS)
wide_scan_downsweep_kernel(const uint32_t *__restrict__ in, uint32_t n, const unsigned long long *__restrict__ tile_offsets,
                           uint64_t *__restrict__ out) {
    __shared__ unsigned long long ws[WS_THREADS / 32 + 1];
    const uint64_t base = (uint64_t)blockIdx.x * WS_TILE + (uint64_t)threadIdx.x * WS_IPT;
    uint32_t v[WS_IPT];
    unsigned long long s = 0;
#pragma unroll
    for (int i = 0; i < WS_IPT; ++i) {
        v[i] = base + i < n ? in[base + i] : 0u;
        s += v[i];
    }
    unsigned long long run = wide_block_scan(s, ws, nullptr) + tile_offsets[blockIdx.x];
#pragma unroll
    for (int i = 0; i < WS_IPT; ++i) {
        if (base + i < n) out[base + i] = run;
        run += v[i];
    }
    if (n > 0 && base <= (uint64_t)n - 1 && (uint64_t)n - 1 < base + WS_IPT) out[n] = run;
}

}  // namespace

void wide_exclusive_scan(spl_ctx *ctx, const uint32_t *in, uint32_t n, uint64_t *out) {
    const unsigned tiles = div_up(n, WS_TILE);
    Tmp<unsigned long long> sums(ctx, tiles + 1);
    wide_scan_reduce_kernel<<<tiles, WS_THREADS, 0, ctx->stream>>>(in, n, sums);
    check_launch(ctx, "wide_scan_reduce");
    wide_scan_spine_kernel<<<1, 1024, 0, ctx->stream>>>(sums, tiles);
    check_launch(ctx, "wide_scan_spine");
    wide_scan_downsweep_kernel<<<tiles, WS_THREADS, 0, ctx->stream>>>(in, n, sums, out);
    check_launch(ctx, "wide_scan_downsweep");
}

uint32_t wide_max_u32(spl_ctx *ctx, const uint32_t *a, uint32_t n) {
    if (n == 0) return 0;
    const unsigned sgrid = (unsigned)ctx->num_sms * 16u;
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, sizeof(uint32_t), ctx->stream));
    wide_max_kernel<<<std::min<unsigned>(div_up(n, 256), sgrid), 256, 0, ctx->stream>>>(a, n, ctx->d_scratch);
    check_launch(ctx, "wide_max");
    uint32_t m = 0;
    read_back(ctx, ctx->d_scratch, &m, 1);
    return m;
}

namespace {

template <typename VB, int LPR>
__global__ void __launch_bounds__(256)
wide_minor_scatter_kernel(const uint64_t *__restrict__ ptr, const uint32_t *__restrict__ ind, const VB *__restrict__ val,
                          uint32_t nmajor, const uint64_t *__restrict__ out_ptr, uint32_t *__restrict__ remaining,
                          uint32_t *__restrict__ out_ind, VB *__restrict__ out_val) {
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t m = gtid / LPR;
    if (m >= nmajor) return;
    const uint64_t e = __ldg(ptr + m + 1);
    for (uint64_t p = __ldg(ptr + m) + (gtid % LPR); p < e; p += LPR) {
        const uint32_t c = __ldg(ind + p);
        const VB v = __ldg(val + p);
        const uint64_t slot = __ldg(out_ptr + c) + atomicSub(remaining + c, 1u) - 1u;
        out_ind[slot] = (uint32_t)m;
        out_val[slot] = v;
    }
}

// LPS lanes own one output segment of at most EPL*LPS entries and put it in ascending major order
// (the order of the reference's row-major sweep; majors are distinct inside a segment)
template <typename VB, int LPS, int EPL>
__global__ void __launch_bounds__(256)
wide_segment_repair_kernel(const uint64_t *__restrict__ out_ptr, uint32_t nseg, uint32_t *__restrict__ out_ind,
                           VB *__restrict__ out_val) {
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t seg = gtid / LPS;
    const unsigned sub = (unsigned)(gtid % LPS);
    const unsigned group_base = lane_id() - sub;
    uint64_t lo = 0;
    uint32_t len = 0;
    if (seg < nseg) {
        lo = __ldg(out_ptr + seg);
        len = (uint32_t)(__ldg(out_ptr + seg + 1) - lo);
    }
    uint32_t r[EPL];
    VB v[EPL];
#pragma unroll
    for (int u = 0; u < EPL; ++u) {
        const uint32_t e = sub + u * LPS;
        r[u] = 0xffffffffu;
        v[u] = VB{};
        if (e < len) { r[u] = out_ind[lo + e]; v[u] = out_val[lo + e]; }
    }
    uint32_t rank[EPL];
#pragma unroll
    for (int u = 0; u < EPL; ++u) rank[u] = 0;
#pragma unroll
    for (int u2 = 0; u2 < EPL; ++u2) {
#pragma unroll 8
        for (int t = 0; t < LPS; ++t) {
            const uint32_t other = __shfl_sync(0xffffffffu, r[u2], group_base + t);
#pragma unroll
            for (int u = 0; u < EPL; ++u) rank[u] += other < r[u];
        }
    }
    __syncwarp();
#pragma unroll
    for (int u = 0; u < EPL; ++u) {
        const uint32_t e = sub + u * LPS;
        if (e < len) { out_ind[lo + rank[u]] = r[u]; out_val[lo + rank[u]] = v[u]; }
    }
}

template <typename VB>
void wide_recompress_t(spl_ctx *ctx, const spl_mat *in, spl_mat *out) {
    const uint32_t nmajor = in->nmajor(), nminor = in->nminor();
    const uint64_t nnz = in->nnz64;
    const unsigned sgrid = (unsigned)ctx->num_sms * 16u;
    Tmp<uint32_t> counts(ctx, nminor);
    SPL_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * (size_t)nminor, ctx->stream));
    wide_minor_count_kernel<<<sgrid, 256, 0, ctx->stream>>>(in->ind, nnz, counts);
    check_launch(ctx, "wide_minor_count");
    const uint32_t longest = wide_max_u32(ctx, counts, nminor);
    SPL_REQUIRE(longest <= kWideRepairMax, SPL_ERR_UNSUPPORTED,
                "transpose of a matrix with 2^32 or more entries: output segments longer than 256 entries are not supported");
    wide_exclusive_scan(ctx, counts, nminor, out->ptr64);
    const VB *val = static_cast<const VB *>(in->val);
    VB *oval = static_cast<VB *>(out->val);
    const double mean = (double)nnz / nmajor;
    auto scatter = [&](auto lpr) {
        constexpr int L = decltype(lpr)::value;
        wide_minor_scatter_kernel<VB, L><<<div_up((uint64_t)nmajor * L, 256), 256, 0, ctx->stream>>>(
            in->ptr64, in->ind, val, nmajor, out->ptr64, counts, out->ind, oval);
    };
    if (mean <= 2.0) scatter(std::integral_constant<int, 1>{});
    else if (mean <= 12.0) scatter(std::integral_constant<int, 4>{});
    else if (mean <= 64.0) scatter(std::integral_constant<int, 8>{});
    else scatter(std::integral_constant<int, 32>{});
    check_launch(ctx, "wide_minor_scatter");
    if (longest > 1) {
        if (longest <= 16)
            wide_segment_repair_kernel<VB, 8, 2><<<div_up((uint64_t)nminor * 8, 256), 256, 0, ctx->stream>>>(out->ptr64, nminor, out->ind, oval);
        else if (longest <= 32)
            wide_segment_repair_kernel<VB, 16, 2><<<div_up((uint64_t)nminor * 16, 256), 256, 0, ctx->stream>>>(out->ptr64, nminor, out->ind, oval);
        else if (longest <= 64)
            wide_segment_repair_kernel<VB, 32, 2><<<div_up((uint64_t)nminor * 32, 256), 256, 0, ctx->stream>>>(out->ptr64, nminor, out->ind, oval);
        else if (longest <= 128)
            wide_segment_repair_kernel<VB, 32, 4><<<div_up((uint64_t)nminor * 32, 256), 256, 0, ctx->stream>>>(out->ptr64, nminor, out->ind, oval);
        else
            wide_segment_repair_kernel<VB, 32, 8><<<div_up((uint64_t)nminor * 32, 256), 256, 0, ctx->stream>>>(out->ptr64, nminor, out->ind, oval);
        check_launch(ctx, "wide_segment_repair");
    }
}

__global__ void __launch_bounds__(256)
wide_entry_range_kernel(const uint64_t *__restrict__ ptr, const uint32_t *__restrict__ ind, uint32_t nmajor, uint64_t start,
                        uint32_t count, uint64_t *__restrict__ major_out, uint64_t *__restrict__ minor_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint64_t p = start + i;
    major_out[i] = upper_bound_u64(ptr, 0, (uint64_t)nmajor + 1, p) - 1;
    minor_out[i] = ind[p];
}

}  // namespace

// SPL_WIDE_MIN_NNZ=<n>: matrices with n stored entries or more are created wide (tests of the wide kernels at
// small sizes), n clamped to [1, 2^32 - 65536]; 2^32 - 65536 when unset or not a number.
uint64_t wide_min_nnz() {
    unsigned long long v = 0;
    if (!env_u64("SPL_WIDE_MIN_NNZ", &v)) return kMaxEntries;
    return v < 1 ? 1 : (v >= kMaxEntries ? kMaxEntries : (uint64_t)v);
}

spl_mat *new_wide_mat(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols, uint64_t nnz) {
    spl_mat *m = new spl_mat();
    m->format = format;
    m->dtype = dtype;
    m->nrows = nrows;
    m->ncols = ncols;
    m->nnz = 0xffffffffu;                    // every 32-bit path refuses a wide matrix before it looks at this
    m->nnz64 = nnz;
    try {
        m->ptr64 = dalloc<uint64_t>(ctx, (size_t)m->nmajor() + 1 + 4);
        m->ind = dalloc<uint32_t>(ctx, (size_t)nnz + 16);
        m->val = dalloc_bytes(ctx, ((size_t)nnz + 16) * m->vsize());
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    return m;
}

int wide_validate(spl_ctx *ctx, const spl_mat *m) {
    const uint32_t nmajor = m->nmajor(), nminor = m->nminor();
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0xff, sizeof(uint32_t), ctx->stream));
    wide_validate_ptr_kernel<<<div_up(nmajor, 256), 256, 0, ctx->stream>>>(m->ptr64, nmajor, ctx->d_scratch);
    check_launch(ctx, "wide_validate_ptr");
    uint32_t fail = 0xffffffffu;
    read_back(ctx, ctx->d_scratch, &fail, 1);
    if (fail != 0xffffffffu) return (int)fail;
    unsigned long long *counters = reinterpret_cast<unsigned long long *>(ctx->d_scratch + 2);
    SPL_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned long long), ctx->stream));
    wide_validate_ind_kernel<<<(unsigned)ctx->num_sms * 16u, 256, 0, ctx->stream>>>(m->ptr64, m->ind, nmajor, nminor, m->nnz64,
                                                                                   ctx->d_scratch, counters);
    check_launch(ctx, "wide_validate_ind");
    uint32_t w[6];
    read_back(ctx, ctx->d_scratch, w, 6);
    if (w[0] != 0xffffffffu) return (int)w[0];
    return (w[2] == w[4] && w[3] == w[5]) ? 0 : 9;
}

void wide_spmv(spl_ctx *ctx, const spl_mat *a, const void *x, void *y) {
    SPL_REQUIRE(a->format == SPL_CSR, SPL_ERR_UNSUPPORTED,
                "SpMV on a CSC matrix with 2^32 or more entries: convert it to CSR first (spl_mat_convert)");
    if (a->dtype == SPL_F32) wide_spmv_t<float>(ctx, a, (const float *)x, (float *)y);
    else wide_spmv_t<double>(ctx, a, (const double *)x, (double *)y);
}

spl_mat *wide_regroup(spl_ctx *ctx, const spl_mat *in, int out_format, uint32_t out_rows, uint32_t out_cols) {
    spl_mat *m = new_wide_mat(ctx, out_format, in->dtype, out_rows, out_cols, in->nnz64);
    try {
        if (in->dtype == SPL_F32) wide_recompress_t<uint32_t>(ctx, in, m);
        else wide_recompress_t<uint64_t>(ctx, in, m);
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    return m;
}

void wide_entry_range(spl_ctx *ctx, const spl_mat *m, uint64_t start, uint32_t count, uint64_t *major_out,
                      uint64_t *minor_out) {
    if (count == 0) return;
    wide_entry_range_kernel<<<div_up(count, 256), 256, 0, ctx->stream>>>(m->ptr64, m->ind, m->nmajor(), start, count,
                                                                        major_out, minor_out);
    check_launch(ctx, "wide_entry_range");
}

}  // namespace spl
