// wide_assemble.cu — COO -> CSR / CSC assembly of 2^32 - 65536 triplets or more.
//
// The reference indexes with usize (src/csr/conv/coo.rs:3-116), so its assembly takes lists of any
// length.  The device assembly (assemble.cu) uses 32-bit positions.  A longer list is cut along the
// major axis (rows for CSR, columns for CSC) into buckets of whole majors, each short enough for that
// assembly, and the parts are stitched:
//   1. one pass over the indices: the bounds of CooMatrix::push (src/coo.rs:432-433) and the number of
//      triplets per major; its 64-bit exclusive scan (wide.cu) gives every major's triplet range;
//   2. the major axis is cut greedily into ranges [m0, m1) of at most B triplets (a longer major is a
//      bucket of its own);
//   3. per bucket, a stable compaction copies the bucket's triplets, in input order, into a scratch
//      list with the major rebased to major - m0: per-tile counts, their scan, a scatter ranked by warp
//      ballots.  Buckets hold whole majors, so every duplicate of a cell lands in one bucket, in
//      insertion order: the in-order sum of the reference is unchanged;
//   4. assemble_from_coo_dev on the scratch list, an (m1 - m0) x nminor problem;
//   5. once every part's nnz is known, the exact-size output (wide if it keeps 2^32 - 65536 entries
//      or more), one kernel for the pointer array, one device copy per part for indices and values;
//      each part is freed as soon as it is copied.
// The compaction reads the input once per bucket instead of partitioning it once into a second full
// copy: at 4.4 G f32 triplets that copy would be 52 GB more than the input itself.
//
// Device memory: B is derived from what is free at the start of the call (step 2).  The peak while the
// buckets run is the input + one bucket's scratch (compacted triplets, the sort's two key/value pairs,
// its part) + the parts so far; at the stitch it is the input + all parts + the output.
#include <algorithm>
#include <vector>

#include "kernels.cuh"

namespace spl {

namespace {

constexpr int WA_THREADS = 256, WA_IPT = 16, WA_TILE = WA_THREADS * WA_IPT;

// Bounds of every triplet and triplets per major (counted only for triplets inside the matrix).
__global__ void __launch_bounds__(256)
wide_coo_scan_kernel(const uint32_t *__restrict__ major, const uint32_t *__restrict__ minor, uint64_t n,
                     uint32_t nmajor, uint32_t nminor, uint32_t *__restrict__ counts, uint32_t *flag) {
    uint32_t bad = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t mj = major[i], mn = minor[i];
        const bool out = (mj >= nmajor) | (mn >= nminor);
        bad |= out;
        if (!out) atomicAdd(counts + mj, 1u);
    }
    if (__any_sync(0xffffffffu, bad) && lane_id() == 0) atomicOr(flag, 1u);
}

// Greedy cut of [0, nmajor) into buckets of at most bmax triplets (one thread: a few binary searches per
// bucket).  cut_major[0..nb] are the bucket bounds, cut_pos[b] = mptr[cut_major[b]].
__global__ void wide_bucket_cut_kernel(const uint64_t *__restrict__ mptr, uint32_t nmajor, uint64_t bmax, uint32_t cap,
                                       uint32_t *__restrict__ cut_major, uint64_t *__restrict__ cut_pos,
                                       uint32_t *__restrict__ count) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    uint32_t m0 = 0, nb = 0;
    cut_major[0] = 0;
    cut_pos[0] = 0;
    while (m0 < nmajor && nb < cap) {
        // last m1 in (m0, nmajor] with mptr[m1] - mptr[m0] <= bmax; m0 + 1 when major m0 alone is longer
        uint64_t m1 = upper_bound_u64(mptr, (uint64_t)m0 + 1, (uint64_t)nmajor + 1, mptr[m0] + bmax) - 1;
        if (m1 <= m0) m1 = (uint64_t)m0 + 1;
        ++nb;
        cut_major[nb] = (uint32_t)m1;
        cut_pos[nb] = mptr[m1];
        m0 = (uint32_t)m1;
    }
    *count = nb;
}

// Compaction, pass 1: triplets of the bucket per tile.  Tiles are WA_THREADS x WA_IPT consecutive
// triplets, warp-striped as in assemble.cu's compact_kernel.
__global__ void __launch_bounds__(WA_THREADS)
wide_bucket_count_kernel(const uint32_t *__restrict__ major, uint64_t n, uint32_t m0, uint32_t span,
                         uint32_t *__restrict__ tile_counts) {
    __shared__ uint32_t ws[WA_THREADS / 32 + 1];
    const uint64_t base = (uint64_t)blockIdx.x * WA_TILE + threadIdx.x;
    uint32_t mj[WA_IPT];
#pragma unroll
    for (int i = 0; i < WA_IPT; ++i) {
        const uint64_t idx = base + (uint64_t)i * WA_THREADS;
        mj[i] = idx < n ? major[idx] - m0 : 0xffffffffu;
    }
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < WA_IPT; ++i) c += mj[i] < span;      // major in [m0, m0 + span): unsigned wrap below m0
    uint32_t total;
    block_exclusive_scan(c, ws, &total);
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

// Compaction, pass 2: the bucket's triplets to scratch position tile offset + rank inside the tile, the
// rank from one ballot per (step, warp) and a scan of the 128 counts: input order is kept.
template <typename VB>
__global__ void __launch_bounds__(WA_THREADS)
wide_bucket_scatter_kernel(const uint32_t *__restrict__ major, const uint32_t *__restrict__ minor,
                           const VB *__restrict__ val, uint64_t n, uint32_t m0, uint32_t span,
                           const uint64_t *__restrict__ tile_offsets, uint32_t *__restrict__ out_major,
                           uint32_t *__restrict__ out_minor, VB *__restrict__ out_val) {
    constexpr int W = WA_THREADS / 32;
    __shared__ uint32_t s_cnt[WA_IPT * W];                    // selected triplets before each (step, warp)
    __shared__ uint32_t s_bal[WA_IPT * W];                    // selected lanes of each (step, warp)
    const uint64_t tile_base = (uint64_t)blockIdx.x * WA_TILE;
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
    uint32_t mj[WA_IPT], mn[WA_IPT];
    VB v[WA_IPT];
    uint32_t sel = 0;
#pragma unroll
    for (int i = 0; i < WA_IPT; ++i) {
        const uint64_t idx = tile_base + (uint64_t)i * WA_THREADS + threadIdx.x;
        mj[i] = idx < n ? major[idx] - m0 : 0xffffffffu;
    }
#pragma unroll
    for (int i = 0; i < WA_IPT; ++i) {
        const uint64_t idx = tile_base + (uint64_t)i * WA_THREADS + threadIdx.x;
        const bool s = mj[i] < span;
        sel |= (uint32_t)s << i;
        mn[i] = s ? minor[idx] : 0u;
        v[i] = s ? val[idx] : VB{};
    }
#pragma unroll
    for (int i = 0; i < WA_IPT; ++i) {
        const unsigned bal = __ballot_sync(0xffffffffu, (sel >> i) & 1u);
        if (lane == 0) { s_cnt[i * W + warp] = __popc(bal); s_bal[i * W + warp] = bal; }
    }
    __syncthreads();
    if (warp == 0) {                       // exclusive scan of the WA_IPT * W (= 128) counts: 4 per lane
        constexpr int PER = WA_IPT * W / 32;
        uint32_t c[PER], sum = 0;
#pragma unroll
        for (int q = 0; q < PER; ++q) { c[q] = s_cnt[lane * PER + q]; sum += c[q]; }
        uint32_t run = warp_inclusive_scan(sum) - sum;
#pragma unroll
        for (int q = 0; q < PER; ++q) { s_cnt[lane * PER + q] = run; run += c[q]; }
    }
    __syncthreads();
    const uint32_t off = (uint32_t)tile_offsets[blockIdx.x];       // < bucket length < 2^32 - 65536
#pragma unroll
    for (int i = 0; i < WA_IPT; ++i) {
        if ((sel >> i) & 1u) {
            const uint32_t pos = off + s_cnt[i * W + warp] + __popc(s_bal[i * W + warp] & lanemask_lt());
            out_major[pos] = mj[i];
            out_minor[pos] = mn[i];
            out_val[pos] = v[i];
        }
    }
}

// The pointer array of the stitched matrix: part j covers majors [cut_major[j], cut_major[j + 1]) and
// starts at entry part_off[j].
template <typename P>
__global__ void __launch_bounds__(256)
wide_stitch_ptr_kernel(const uint32_t *const *__restrict__ part_ptr, const uint64_t *__restrict__ part_off,
                       const uint32_t *__restrict__ cut_major, uint32_t nparts, uint32_t nmajor, uint64_t total,
                       P *__restrict__ out) {
    const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m > nmajor) return;
    if (m == nmajor) { out[m] = (P)total; return; }
    const uint32_t j = upper_bound_u32(cut_major, 0, nparts + 1, (uint32_t)m) - 1;
    out[m] = (P)(part_off[j] + part_ptr[j][m - cut_major[j]]);
}

// Bucket bound: the free device memory (plus what the library's pool holds idle) at the start of the
// call, minus room for the parts (at most every triplet survives: 4 + V bytes each) and the histogram,
// over the scratch one bucket triplet needs: the compacted triplet (8 + V), the two key/value pairs of
// the sort (2 (K + V)), the tail's flag and slack (2), the bucket's part (4 + V).  10 % is held back
// for the pool's rounding and the sort's small arrays.
uint64_t bucket_bound(spl_ctx *ctx, uint64_t len, uint32_t nmajor, int key_bytes, size_t vs) {
    size_t free_b = 0, total_b = 0;
    SPL_CUDA(cudaMemGetInfo(&free_b, &total_b));
    uint64_t reserved = 0, used = 0;
    SPL_CUDA(cudaMemPoolGetAttribute(ctx->pool, cudaMemPoolAttrReservedMemCurrent, &reserved));
    SPL_CUDA(cudaMemPoolGetAttribute(ctx->pool, cudaMemPoolAttrUsedMemCurrent, &used));
    const double avail = 0.9 * ((double)free_b + (double)(reserved > used ? reserved - used : 0));
    const double parts = (double)len * (4 + vs) + (double)nmajor * 16;
    const double per = (double)(8 + vs) + 2.0 * (key_bytes + vs) + 2.0 + (double)(4 + vs);
    const double b = (avail - parts) / per;
    const uint64_t floor_b = 1ull << 24;                        // below this, the allocations decide (SPL_ERR_OOM)
    const uint64_t cap_b = kMaxEntries - 1;
    if (!(b > (double)floor_b)) return floor_b;
    return b >= (double)cap_b ? cap_b : (uint64_t)b;
}

// Parts owned until they are copied into the output; freed on every path.
struct Parts {
    spl_ctx *ctx;
    std::vector<spl_mat *> m;
    explicit Parts(spl_ctx *c) : ctx(c) {}
    ~Parts() {
        for (spl_mat *p : m) free_mat(ctx, p);
    }
};

template <typename VB>
spl_mat *assemble_bucketed(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols, uint64_t len,
                           const uint32_t *major_idx, const uint32_t *minor_idx, const VB *val, int dedup,
                           int dropzero, uint64_t bmax) {
    const bool csr = format == SPL_CSR;
    const uint32_t nmajor = csr ? nrows : ncols, nminor = csr ? ncols : nrows;
    const unsigned sgrid = (unsigned)ctx->num_sms * 16u;
    // 1. bounds and the major histogram, then the triplet range of every major
    Tmp<uint64_t> mptr(ctx, (size_t)nmajor + 1);
    {
        Tmp<uint32_t> counts(ctx, nmajor);
        SPL_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * (size_t)nmajor, ctx->stream));
        SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, sizeof(uint32_t), ctx->stream));
        const unsigned g = div_up(len, 256 * 8);
        wide_coo_scan_kernel<<<g < sgrid ? g : sgrid, 256, 0, ctx->stream>>>(major_idx, minor_idx, len, nmajor, nminor,
                                                                           counts, ctx->d_scratch);
        check_launch(ctx, "wide_coo_scan");
        uint32_t bad = 0;
        read_back(ctx, ctx->d_scratch, &bad, 1);
        SPL_REQUIRE(bad == 0, SPL_ERR_ARG, "COO entry out of bounds (CooMatrix::push asserts row < nrows, col < ncols)");
        const uint32_t longest = wide_max_u32(ctx, counts, nmajor);
        wide_exclusive_scan(ctx, counts, nmajor, mptr);
        uint32_t tw[2] = {0, 0};
        read_back(ctx, reinterpret_cast<const uint32_t *>(mptr.p + nmajor), tw, 2);
        // a count that wrapped (2^32 triplets or more in one major) shows as a total below len
        SPL_REQUIRE(((uint64_t)tw[1] << 32 | tw[0]) == len && longest < kMaxEntries, SPL_ERR_UNSUPPORTED,
                    csr ? "COO assembly: one row holds 2^32 - 65536 triplets or more (at most 2^32 - 65537 per row)"
                        : "COO assembly: one column holds 2^32 - 65536 triplets or more (at most 2^32 - 65537 per column)");
    }
    // 2. buckets of whole majors
    const uint64_t cap64 = 2 * (len / bmax) + 3;               // two neighbouring buckets hold more than bmax
    const uint32_t cap = (uint32_t)std::min<uint64_t>(cap64, (uint64_t)nmajor);
    Tmp<uint32_t> cut_major(ctx, (size_t)cap + 1);
    Tmp<uint64_t> cut_pos(ctx, (size_t)cap + 1);
    wide_bucket_cut_kernel<<<1, 32, 0, ctx->stream>>>(mptr, nmajor, bmax, cap, cut_major, cut_pos, ctx->d_scratch);
    check_launch(ctx, "wide_bucket_cut");
    uint32_t nb = 0;
    read_back(ctx, ctx->d_scratch, &nb, 1);
    std::vector<uint32_t> h_major((size_t)nb + 1);
    std::vector<uint64_t> h_pos((size_t)nb + 1);
    SPL_CUDA(cudaMemcpyAsync(h_major.data(), cut_major, sizeof(uint32_t) * (nb + 1), cudaMemcpyDeviceToHost, ctx->stream));
    SPL_CUDA(cudaMemcpyAsync(h_pos.data(), cut_pos, sizeof(uint64_t) * (nb + 1), cudaMemcpyDeviceToHost, ctx->stream));
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    SPL_REQUIRE(h_major[nb] == nmajor && h_pos[nb] == len, SPL_ERR_CUDA, "COO assembly: bucket cut incomplete");
    // 3 + 4. per bucket: stable compaction, then the 32-bit assembly
    const uint64_t tiles64 = (len + WA_TILE - 1) / WA_TILE;
    const uint32_t tiles = (uint32_t)tiles64;
    Parts parts(ctx);
    parts.m.reserve(nb);
    {
        Tmp<uint32_t> tile_counts(ctx, tiles);
        Tmp<uint64_t> tile_offsets(ctx, (size_t)tiles + 1);
        for (uint32_t b = 0; b < nb; ++b) {
            const uint32_t m0 = h_major[b], span = h_major[b + 1] - m0;
            const uint64_t blen = h_pos[b + 1] - h_pos[b];       // < kMaxEntries: no major is that long
            Tmp<uint32_t> bmaj(ctx, blen), bmin(ctx, blen);
            Tmp<VB> bval(ctx, blen);
            if (blen) {
                wide_bucket_count_kernel<<<tiles, WA_THREADS, 0, ctx->stream>>>(major_idx, len, m0, span, tile_counts);
                check_launch(ctx, "wide_bucket_count");
                wide_exclusive_scan(ctx, tile_counts, tiles, tile_offsets);
                wide_bucket_scatter_kernel<VB><<<tiles, WA_THREADS, 0, ctx->stream>>>(
                    major_idx, minor_idx, val, len, m0, span, tile_offsets, bmaj, bmin, bval);
                check_launch(ctx, "wide_bucket_scatter");
            }
            const uint32_t *brow = csr ? bmaj.p : bmin.p, *bcol = csr ? bmin.p : bmaj.p;
            parts.m.push_back(assemble_from_coo_dev(ctx, format, dtype, csr ? span : nrows, csr ? ncols : span,
                                                   (uint32_t)blen, brow, bcol, bval.p, dedup, dropzero));   // reserved: no throw
        }
    }
    // 5. stitch
    std::vector<uint64_t> h_off((size_t)nb + 1, 0);
    std::vector<const uint32_t *> h_ptr(nb);
    for (uint32_t b = 0; b < nb; ++b) {
        h_off[b + 1] = h_off[b] + parts.m[b]->nnz;
        h_ptr[b] = parts.m[b]->ptr;
    }
    const uint64_t total = h_off[nb];
    spl_mat *out = total >= wide_min_nnz() ? new_wide_mat(ctx, format, dtype, nrows, ncols, total)
                                        : new_mat(ctx, format, dtype, nrows, ncols, (uint32_t)total);
    try {
        {
            Tmp<const uint32_t *> d_ptr(ctx, nb);
            Tmp<uint64_t> d_off(ctx, nb);
            SPL_CUDA(cudaMemcpyAsync(d_ptr.p, h_ptr.data(), sizeof(const uint32_t *) * nb, cudaMemcpyHostToDevice, ctx->stream));
            SPL_CUDA(cudaMemcpyAsync(d_off.p, h_off.data(), sizeof(uint64_t) * nb, cudaMemcpyHostToDevice, ctx->stream));
            const unsigned g = div_up((uint64_t)nmajor + 1, 256);
            if (out->wide())
                wide_stitch_ptr_kernel<uint64_t><<<g, 256, 0, ctx->stream>>>(d_ptr, d_off, cut_major, nb, nmajor, total,
                                                                           out->ptr64);
            else
                wide_stitch_ptr_kernel<uint32_t><<<g, 256, 0, ctx->stream>>>(d_ptr, d_off, cut_major, nb, nmajor, total,
                                                                           out->ptr);
            check_launch(ctx, "wide_stitch_ptr");
            // the pageable sources of the two table uploads must outlive them
            SPL_CUDA(cudaStreamSynchronize(ctx->stream));
        }
        for (uint32_t b = 0; b < nb; ++b) {
            spl_mat *p = parts.m[b];
            if (p->nnz) {
                SPL_CUDA(cudaMemcpyAsync(out->ind + h_off[b], p->ind, sizeof(uint32_t) * (size_t)p->nnz,
                                         cudaMemcpyDeviceToDevice, ctx->stream));
                SPL_CUDA(cudaMemcpyAsync(static_cast<VB *>(out->val) + h_off[b], p->val, sizeof(VB) * (size_t)p->nnz,
                                         cudaMemcpyDeviceToDevice, ctx->stream));
            }
            parts.m[b] = nullptr;
            free_mat(ctx, p);                                         // stream-ordered: after its copies
        }
    } catch (...) {
        free_mat(ctx, out);
        throw;
    }
    return out;
}

// SPL_ASSEMBLE_BUCKET_MAX=<triplets>: lists longer than that take the bucketed route with buckets of at
// most that many triplets (tests of the route at small sizes); 0 when unset or not a number.
uint64_t bucket_knob() {
    unsigned long long v = 0;
    if (!env_u64("SPL_ASSEMBLE_BUCKET_MAX", &v)) return 0;
    return v < 1 ? 1 : (v >= kMaxEntries ? kMaxEntries - 1 : (uint64_t)v);
}

}  // namespace

bool assemble_is_bucketed(uint64_t len) {
    const uint64_t knob = bucket_knob();
    return len >= kMaxEntries || (knob && len > knob);
}

spl_mat *assemble_from_coo_any(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols,
                               uint64_t len, const uint32_t *row, const uint32_t *col,
                               const void *val, int dedup, int dropzero) {
    if (!assemble_is_bucketed(len))
        return assemble_from_coo_dev(ctx, format, dtype, nrows, ncols, (uint32_t)len, row, col, val, dedup, dropzero);
    const bool csr = format == SPL_CSR;
    const uint32_t nmajor = csr ? nrows : ncols;
    const size_t vs = dtype == SPL_F32 ? 4 : 8;
    uint64_t bmax = bucket_knob();
    if (!bmax || len <= bmax) {
        const int key_bytes = bits_for(nrows) + bits_for(ncols) > 32 ? 8 : 4;
        bmax = bucket_bound(ctx, len, nmajor, key_bytes, vs);
    }
    const uint32_t *major = csr ? row : col, *minor = csr ? col : row;
    if (dtype == SPL_F32)
        return assemble_bucketed<uint32_t>(ctx, format, dtype, nrows, ncols, len, major, minor,
                                           static_cast<const uint32_t *>(val), dedup, dropzero, bmax);
    return assemble_bucketed<uint64_t>(ctx, format, dtype, nrows, ncols, len, major, minor,
                                       static_cast<const uint64_t *>(val), dedup, dropzero, bmax);
}

}  // namespace spl
