// gather_rows.cu — the exchange of the row-sharded sparse product (spl_peer_gather_rows).
//
// C = A * B with A, B sharded by rows across the ranks of one box: rank g's rows of C need exactly the rows of B
// that the stored columns of its rows of A name.  This file copies those rows, wherever they live, into one ordinary
// local matrix of B's full height (every other row empty), so that the single-GPU spgemm multiplies A's shard by it
// unchanged: each C[i,j] still sums over ascending k, bit for bit the unsharded product.  The same code serves the
// column-sharded CSC twin (majors = columns).
//
// Device passes (one host synchronisation, to size the output exactly):
//   mark    flag every major that one of by's stored minor indices names;
//   count   length of every marked major, read from its owner's pointer array over peer memory (checked against
//           the owner's entry count, so a corrupt pointer never becomes an out-of-range peer read), 64-bit total;
//   flag    first major of every run: a run is a maximal range of consecutive non-empty marked majors with one owner,
//           i.e. one contiguous range of the owner's ind / val and one contiguous range of the output;
//   scans   exclusive_scan_u32 of the counts is the output's full-height pointer array, of the flags the run ids;
//   runs    compact the runs (output position, owner position, owner);
//   copy    long runs (>= GR_LONG entries) through TMA bulk copies into a shared-memory ring, the CTA storing each
//           stage at the element shift between source and output; short runs (random matrices: mostly one row)
//           through loads spread over the output, four per array in flight per thread.
#include <algorithm>

#include "kernels.cuh"
#include "ptx.cuh"
#include "scan.cuh"

namespace spl {

namespace {

struct GatherShards {
    const uint32_t *ptr[SPL_MAX_PEERS];
    const unsigned char *ind[SPL_MAX_PEERS];
    const unsigned char *val[SPL_MAX_PEERS];
    uint32_t start[SPL_MAX_PEERS + 1];
    uint32_t nnz[SPL_MAX_PEERS];
    int world;
};

// A run this long or longer is copied by the bulk-copy kernel: below one ring chunk of indices (16 KB) a TMA round
// trip moves less than the loads of the short path keep in flight for the same run.
constexpr uint32_t GR_LONG = 4096;
constexpr uint32_t GR_CHUNK = 16384;          // bytes of one ring stage
constexpr int GR_STAGES = 4;
constexpr int GR_THREADS = 256;
constexpr int GR_UNROLL = 4;                  // short path: output entries per thread
constexpr uint32_t GR_TILE = GR_THREADS * GR_UNROLL;

__device__ __forceinline__ int owner_of(const GatherShards &s, uint32_t j) {
    int g = 0;
    while (j >= s.start[g + 1]) ++g;          // start[world] = nmajor > j; empty ranks are stepped over
    return g;
}

__global__ void gr_mark_kernel(const uint32_t *__restrict__ ind, uint32_t n, uint8_t *__restrict__ mark) {
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (uint64_t)gridDim.x * blockDim.x)
        mark[ind[p]] = 1;
}

__global__ void __launch_bounds__(256)
gr_count_kernel(GatherShards s, const uint8_t *__restrict__ mark, uint32_t nmajor, uint32_t *__restrict__ count,
                unsigned long long *__restrict__ total, uint32_t *__restrict__ bad) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t c = 0;
    if (j < nmajor) {
        if (mark[j]) {
            const int g = owner_of(s, (uint32_t)j);
            const uint32_t l = (uint32_t)j - s.start[g];
            const uint32_t lo = __ldcg(s.ptr[g] + l), hi = __ldcg(s.ptr[g] + l + 1);
            if (lo <= hi && hi <= s.nnz[g]) c = hi - lo;
            else atomicOr(bad, 1u);
        }
        count[j] = c;
    }
    unsigned long long t = c;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane_id() == 0 && t) atomicAdd(total, t);
}

__global__ void gr_flag_kernel(GatherShards s, const uint32_t *__restrict__ count, uint32_t nmajor,
                               uint32_t *__restrict__ flag) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nmajor) return;
    bool first = count[j] != 0 && (j == 0 || count[j - 1] == 0);
    for (int g = 1; g < s.world; ++g) first |= count[j] != 0 && s.start[g] == j;      // owner boundary
    flag[j] = first;
}

__global__ void gr_runs_kernel(GatherShards s, const uint32_t *__restrict__ flag, const uint32_t *__restrict__ run_id,
                               const uint32_t *__restrict__ cptr, uint32_t nmajor, uint32_t nruns,
                               uint32_t *__restrict__ run_dst, uint32_t *__restrict__ run_src,
                               uint8_t *__restrict__ run_owner) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nmajor) return;
    if (j == 0) run_dst[nruns] = cptr[nmajor];          // runs tile the output: run r ends where r + 1 begins
    if (!flag[j]) return;
    const uint32_t r = run_id[j];
    const int g = owner_of(s, (uint32_t)j);
    run_dst[r] = cptr[j];
    run_src[r] = __ldcg(s.ptr[g] + ((uint32_t)j - s.start[g]));
    run_owner[r] = (uint8_t)g;
}

// the 16-byte aligned window [lo, hi) around `bytes` bytes at `addr`, in whole chunks
__device__ __forceinline__ uint32_t window_chunks(uint64_t addr, uint64_t bytes) {
    const uint64_t lo = addr & ~15ull, hi = (addr + bytes + 15) & ~15ull;
    return (uint32_t)((hi - lo + GR_CHUNK - 1) / GR_CHUNK);
}

// bulk-copy work of every run: chunks of its index window, then chunks of its value window (0 for a short run)
__global__ void gr_items_kernel(GatherShards s, const uint32_t *__restrict__ run_dst,
                                const uint32_t *__restrict__ run_src, const uint8_t *__restrict__ run_owner,
                                uint32_t nruns, uint32_t vsize, uint32_t *__restrict__ items) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nruns) return;
    const uint32_t len = run_dst[r + 1] - run_dst[r];
    uint32_t n = 0;
    if (len >= GR_LONG) {
        const int g = run_owner[r];
        n = window_chunks((uint64_t)(uintptr_t)s.ind[g] + 4ull * run_src[r], 4ull * len) +
            window_chunks((uint64_t)(uintptr_t)s.val[g] + (uint64_t)vsize * run_src[r], (uint64_t)vsize * len);
    }
    items[r] = n;
}

// Short runs.  CTA b owns output positions [b * GR_TILE, (b + 1) * GR_TILE); every run holds an entry, so the
// GR_TILE runs from the one holding the first position cover the tile.  Their descriptors go to shared memory, each
// thread finds the run of its positions there and issues all its loads (indices and values, peer memory) before
// its stores.  Positions of long runs are left to gr_long_kernel.
template <typename V>
__global__ void __launch_bounds__(GR_THREADS)
gr_short_kernel(GatherShards s, const uint32_t *__restrict__ run_dst, const uint32_t *__restrict__ run_src,
                const uint8_t *__restrict__ run_owner, uint32_t nruns, uint32_t total, uint32_t *__restrict__ out_ind,
                V *__restrict__ out_val) {
    __shared__ uint32_t w_dst[GR_TILE + 1], w_src[GR_TILE];
    __shared__ uint8_t w_own[GR_TILE];
    __shared__ uint32_t s_r0;
    const uint32_t p0 = blockIdx.x * GR_TILE;
    if (threadIdx.x == 0) s_r0 = upper_bound_u32(run_dst, 0, nruns + 1, p0) - 1;
    __syncthreads();
    const uint32_t r0 = s_r0, nw = min(GR_TILE, nruns - r0);
    for (uint32_t k = threadIdx.x; k <= nw; k += GR_THREADS) {
        w_dst[k] = run_dst[r0 + k];
        if (k < nw) {
            w_src[k] = run_src[r0 + k];
            w_own[k] = run_owner[r0 + k];
        }
    }
    __syncthreads();
    if (w_dst[1] - w_dst[0] >= GR_LONG && w_dst[1] >= p0 + GR_TILE) return;     // the tile lies in one long run
    uint32_t c[GR_UNROLL];
    V v[GR_UNROLL];
    uint32_t at[GR_UNROLL];
#pragma unroll
    for (int u = 0; u < GR_UNROLL; ++u) {
        const uint32_t p = p0 + u * GR_THREADS + threadIdx.x;
        at[u] = 0xffffffffu;
        if (p >= total) continue;
        uint32_t lo = 0, hi = nw;                       // last run r of the window with w_dst[r] <= p
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (w_dst[mid] <= p) lo = mid;
            else hi = mid;
        }
        if (w_dst[lo + 1] - w_dst[lo] >= GR_LONG) continue;
        const int g = w_own[lo];
        const uint32_t q = w_src[lo] + (p - w_dst[lo]);
        c[u] = __ldcg(reinterpret_cast<const uint32_t *>(s.ind[g]) + q);
        v[u] = __ldcg(reinterpret_cast<const V *>(s.val[g]) + q);
        at[u] = p;
    }
#pragma unroll
    for (int u = 0; u < GR_UNROLL; ++u) {
        if (at[u] == 0xffffffffu) continue;
        out_ind[at[u]] = c[u];
        out_val[at[u]] = v[u];
    }
}

// One bulk-copy chunk: `bytes` (a multiple of 16) from the 16-byte aligned source address `src`, of which the bytes
// in [want_lo, want_hi) go to `dst` + (byte - want_lo); `elem` = 4 (indices) or 8 / 4 (values).
struct GrChunk {
    uint64_t src, want_lo, want_hi;
    unsigned char *dst;
    uint32_t bytes, elem;
};

__device__ __forceinline__ GrChunk gr_locate(const GatherShards &s, const uint32_t *run_dst, const uint32_t *run_src,
                                             const uint8_t *run_owner, const uint32_t *item_off, uint32_t nruns,
                                             uint32_t vsize, uint32_t *out_ind, unsigned char *out_val, uint32_t item) {
    const uint32_t r = upper_bound_u32(item_off, 0, nruns + 1, item) - 1;
    const uint32_t len = run_dst[r + 1] - run_dst[r];
    const int g = run_owner[r];
    uint32_t k = item - item_off[r];
    uint64_t addr = (uint64_t)(uintptr_t)s.ind[g] + 4ull * run_src[r];
    uint64_t bytes = 4ull * len;
    GrChunk c;
    c.dst = reinterpret_cast<unsigned char *>(out_ind + run_dst[r]);
    c.elem = 4;
    const uint32_t nind = window_chunks(addr, bytes);
    if (k >= nind) {
        k -= nind;
        addr = (uint64_t)(uintptr_t)s.val[g] + (uint64_t)vsize * run_src[r];
        bytes = (uint64_t)vsize * len;
        c.dst = out_val + (uint64_t)vsize * run_dst[r];
        c.elem = vsize;
    }
    const uint64_t w0 = addr & ~15ull, w1 = (addr + bytes + 15) & ~15ull;
    c.src = w0 + (uint64_t)k * GR_CHUNK;
    c.bytes = (uint32_t)(w1 - c.src < GR_CHUNK ? w1 - c.src : GR_CHUNK);
    c.want_lo = addr;
    c.want_hi = addr + bytes;
    return c;
}

// Long runs.  Item i = one chunk of a long run's aligned index or value window; CTA b takes items b, b + grid, ...
// Thread 0 keeps GR_STAGES bulk copies in flight (peer memory -> ring, completion on an mbarrier per stage); all
// threads store a landed stage at the element shift between source and output (any multiple of 4 / 8 bytes, so not
// a bulk store), then the stage is refilled.  The aligned window reaches at most 15 bytes beyond the run on either
// side, inside the 16-byte units that hold its first and last byte.
__global__ void __launch_bounds__(GR_THREADS)
gr_long_kernel(GatherShards s, const uint32_t *__restrict__ run_dst, const uint32_t *__restrict__ run_src,
               const uint8_t *__restrict__ run_owner, const uint32_t *__restrict__ item_off, uint32_t nruns,
               uint32_t vsize, uint32_t *__restrict__ out_ind, unsigned char *__restrict__ out_val) {
    extern __shared__ __align__(128) unsigned char gr_ring[];
    __shared__ __align__(8) uint64_t full[GR_STAGES];
    const uint32_t nitems = item_off[nruns];
    if (blockIdx.x >= nitems) return;
    const uint32_t mine = (nitems - blockIdx.x + gridDim.x - 1) / gridDim.x;
    auto locate = [&](uint32_t q) {
        return gr_locate(s, run_dst, run_src, run_owner, item_off, nruns, vsize, out_ind, out_val,
                         blockIdx.x + q * gridDim.x);
    };
    if (threadIdx.x == 0) {
        for (int st = 0; st < GR_STAGES; ++st) mbar_init(full + st, 1);
        mbar_init_fence();
        for (uint32_t q = 0; q < mine && q < (uint32_t)GR_STAGES; ++q) {
            const GrChunk c = locate(q);
            mbar_expect_tx(full + q, c.bytes);
            tma_bulk_g2s(gr_ring + (size_t)q * GR_CHUNK, reinterpret_cast<const void *>(c.src), c.bytes, full + q);
        }
    }
    __syncthreads();
    for (uint32_t q = 0; q < mine; ++q) {
        const int st = (int)(q % GR_STAGES);
        const GrChunk c = locate(q);
        mbar_wait(full + st, (q / GR_STAGES) & 1u);
        const unsigned char *stage = gr_ring + (size_t)st * GR_CHUNK;
        const uint32_t n = c.bytes / c.elem;
        if (c.elem == 8) {
            for (uint32_t e = threadIdx.x; e < n; e += GR_THREADS) {
                const uint64_t b = c.src + 8ull * e;
                if (b >= c.want_lo && b < c.want_hi)
                    reinterpret_cast<unsigned long long *>(c.dst)[(b - c.want_lo) >> 3] =
                        reinterpret_cast<const unsigned long long *>(stage)[e];
            }
        } else {
            for (uint32_t e = threadIdx.x; e < n; e += GR_THREADS) {
                const uint64_t b = c.src + 4ull * e;
                if (b >= c.want_lo && b < c.want_hi)
                    reinterpret_cast<uint32_t *>(c.dst)[(b - c.want_lo) >> 2] = reinterpret_cast<const uint32_t *>(stage)[e];
            }
        }
        fence_proxy_async_smem();
        __syncthreads();                                  // every thread is done with the stage
        if (threadIdx.x == 0 && q + GR_STAGES < mine) {
            const GrChunk nx = locate(q + GR_STAGES);
            mbar_expect_tx(full + st, nx.bytes);
            tma_bulk_g2s(gr_ring + (size_t)st * GR_CHUNK, reinterpret_cast<const void *>(nx.src), nx.bytes, full + st);
        }
    }
}

}  // namespace

spl_mat *peer_gather_rows(spl_ctx *ctx, int format, int dtype, uint32_t nmajor, uint32_t nminor, int world,
                          const uint64_t *starts, const uint64_t *shard_nnz, const void *const *ptr_slices,
                          const void *const *ind_slices, const void *const *val_slices, const spl_mat *by) {
    GatherShards s{};
    s.world = world;
    for (int g = 0; g <= SPL_MAX_PEERS; ++g) s.start[g] = (uint32_t)starts[g < world ? g : world];
    for (int g = 0; g < world; ++g) {
        s.ptr[g] = static_cast<const uint32_t *>(ptr_slices[g]);
        s.ind[g] = static_cast<const unsigned char *>(ind_slices[g]);
        s.val[g] = static_cast<const unsigned char *>(val_slices[g]);
        s.nnz[g] = (uint32_t)shard_nnz[g];
    }
    const uint32_t vsize = dtype == SPL_F32 ? 4u : 8u;
    const unsigned blocks = div_up(nmajor, 256);

    Tmp<uint8_t> mark(ctx, nmajor);
    Tmp<uint32_t> count(ctx, nmajor), flag(ctx, nmajor), run_id(ctx, (size_t)nmajor + 1);
    Tmp<uint32_t> cptr(ctx, (size_t)nmajor + 1 + 4);                // becomes the output's pointer array (new_mat's slack)
    unsigned long long *total64 = reinterpret_cast<unsigned long long *>(ctx->d_scratch + 40);
    uint32_t *bad = ctx->d_scratch + 42;
    SPL_CUDA(cudaMemsetAsync(mark, 0, nmajor, ctx->stream));
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch + 40, 0, 4 * sizeof(uint32_t), ctx->stream));
    if (by->nnz) {
        gr_mark_kernel<<<std::min<unsigned>(div_up(by->nnz, 256), (unsigned)ctx->num_sms * 16u), 256, 0, ctx->stream>>>(
            by->ind, by->nnz, mark);
        check_launch(ctx, "gather_rows_mark");
    }
    gr_count_kernel<<<blocks, 256, 0, ctx->stream>>>(s, mark, nmajor, count, total64, bad);
    check_launch(ctx, "gather_rows_count");
    gr_flag_kernel<<<blocks, 256, 0, ctx->stream>>>(s, count, nmajor, flag);
    check_launch(ctx, "gather_rows_flag");
    exclusive_scan_u32(ctx, count, nmajor, cptr);
    exclusive_scan_u32(ctx, flag, nmajor, run_id);
    SPL_CUDA(cudaMemcpyAsync(ctx->d_scratch + 43, run_id.p + nmajor, sizeof(uint32_t), cudaMemcpyDeviceToDevice,
                             ctx->stream));
    uint32_t w[4];
    read_back(ctx, ctx->d_scratch + 40, w, 4);
    SPL_REQUIRE(w[2] == 0, SPL_ERR_ARG,
                "spl_peer_gather_rows: a shard's pointer array descends or points past its entry count");
    const uint64_t total = (uint64_t)w[0] | ((uint64_t)w[1] << 32);
    SPL_REQUIRE(total < kMaxEntries, SPL_ERR_UNSUPPORTED,
                "spl_peer_gather_rows: the gathered rows hold 2^32 - 65536 entries or more");
    const uint32_t nruns = w[3];

    spl_mat *m = new_mat(ctx, format, dtype, format == SPL_CSR ? nmajor : nminor, format == SPL_CSR ? nminor : nmajor,
                         (uint32_t)total);
    dfree(ctx, m->ptr);
    m->ptr = cptr.release();
    if (!total) return m;
    try {
        Tmp<uint32_t> run_dst(ctx, (size_t)nruns + 1), run_src(ctx, nruns), items(ctx, nruns), item_off(ctx, (size_t)nruns + 1);
        Tmp<uint8_t> run_owner(ctx, nruns);
        gr_runs_kernel<<<blocks, 256, 0, ctx->stream>>>(s, flag, run_id, m->ptr, nmajor, nruns, run_dst, run_src,
                                                        run_owner);
        check_launch(ctx, "gather_rows_runs");
        gr_items_kernel<<<div_up(nruns, 256), 256, 0, ctx->stream>>>(s, run_dst, run_src, run_owner, nruns, vsize, items);
        check_launch(ctx, "gather_rows_items");
        exclusive_scan_u32(ctx, items, nruns, item_off);
        const unsigned tiles = div_up(total, GR_TILE);
        if (dtype == SPL_F32)
            gr_short_kernel<uint32_t><<<tiles, GR_THREADS, 0, ctx->stream>>>(
                s, run_dst, run_src, run_owner, nruns, (uint32_t)total, m->ind, static_cast<uint32_t *>(m->val));
        else
            gr_short_kernel<unsigned long long><<<tiles, GR_THREADS, 0, ctx->stream>>>(
                s, run_dst, run_src, run_owner, nruns, (uint32_t)total, m->ind, static_cast<unsigned long long *>(m->val));
        check_launch(ctx, "gather_rows_short");
        // a grid that exits at once when no run is long (the item count is read on the device)
        const size_t smem = (size_t)GR_CHUNK * GR_STAGES;
        SPL_CUDA(cudaFuncSetAttribute(gr_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        gr_long_kernel<<<(unsigned)ctx->num_sms * 2u, GR_THREADS, smem, ctx->stream>>>(
            s, run_dst, run_src, run_owner, item_off, nruns, vsize, m->ind, static_cast<unsigned char *>(m->val));
        check_launch(ctx, "gather_rows_long");
    } catch (...) {
        free_mat(ctx, m);
        throw;
    }
    return m;
}

}  // namespace spl
