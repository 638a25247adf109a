// peer.cu — peer-visible device memory and a flag barrier over it (SURVEY.md 8e).
//
// One process per GPU.  A rank allocates its slice of x (and a small flag block) with
// cudaMalloc, exports it with CUDA IPC, and maps its peers' blocks; on an NVSwitch box every
// mapping is a full-bandwidth NVLink path.  spl_spmv_peer then gathers x straight from the
// owning slice, so the "exchange" of the sharded SpMV is part of the kernel's loads.  The only
// thing left between iterations is ordering: a rank's writes to its slice must be visible before
// a peer's next kernel reads them.  peer_barrier_kernel does that on the device with the flag
// barrier of ptx.cuh: release-store of the epoch into every peer's flag block, acquire-spin on the
// own block, bounded by a timeout so a missing peer can never hang the GPU.
#include <algorithm>
#include <cstdlib>

#include "kernels.cuh"
#include "ptx.cuh"

namespace spl {

namespace {

struct FlagBlocks {
    uint32_t *block[SPL_MAX_PEERS];
};

__global__ void peer_barrier_kernel(FlagBlocks f, int world, int rank, uint32_t epoch,
                                    uint64_t timeout_ns, uint32_t *timed_out) {
    const int g = threadIdx.x;
    if (g >= world || g == rank) return;
    flag_arrive(f.block[g], rank, epoch);        // earlier kernels' writes to this rank's slice are visible
    flag_wait(f.block[rank] + g, epoch, timeout_ns, 200, timed_out);
}

// Barrier + halo in one launch.  Threads 0..world-1 run the flag protocol above; once every peer has
// arrived, the whole CTA copies this rank's halo — the halo_left columns before and the halo_right
// columns after its own slice — element by element from the owning ranks' slices (peer memory) into
// the padding that surrounds the own slice.  The product that follows then gathers from ONE local
// array (own slice + halo) with the plain local policy: for a banded or stencil shard this moves the
// same few values over NVLink as the in-kernel peer gather, without an owner test on every gather.
struct HaloSlices {
    unsigned char *slice[SPL_MAX_PEERS];
    unsigned long long start[SPL_MAX_PEERS + 1];
    unsigned int halo_left, halo_right, vsize;
};

__global__ void __launch_bounds__(256)
peer_barrier_halo_kernel(FlagBlocks f, int world, int rank, uint32_t epoch, uint64_t timeout_ns, uint32_t *timed_out,
                         HaloSlices h) {
    __shared__ int s_failed;
    if (threadIdx.x == 0) s_failed = 0;
    __syncthreads();
    const int g = threadIdx.x;
    if (g < world && g != rank) {
        flag_arrive(f.block[g], rank, epoch);
        if (!flag_wait(f.block[rank] + g, epoch, timeout_ns, 200, timed_out)) s_failed = 1;
    }
    __syncthreads();
    if (s_failed) return;                        // the product behind this writes NaN (XPeer / status call)
    const unsigned long long my0 = h.start[rank], my1 = h.start[rank + 1], n = h.start[world];
    const unsigned int total = h.halo_left + h.halo_right;
    for (unsigned int i = threadIdx.x; i < total; i += blockDim.x) {
        long long col = i < h.halo_left ? (long long)my0 - h.halo_left + i : (long long)my1 + (i - h.halo_left);
        if (col < 0 || (unsigned long long)col >= n) continue;
        int owner = 0;
        for (int q = 0; q < world; ++q)
            if ((unsigned long long)col >= h.start[q] && (unsigned long long)col < h.start[q + 1]) owner = q;
        const unsigned char *src = h.slice[owner] + ((unsigned long long)col - h.start[owner]) * h.vsize;
        unsigned char *dst = h.slice[rank] + (col - (long long)my0) * (long long)h.vsize;     // before / after the own slice
        if (h.vsize == 8) *reinterpret_cast<unsigned long long *>(dst) = __ldcg(reinterpret_cast<const unsigned long long *>(src));
        else *reinterpret_cast<unsigned int *>(dst) = __ldcg(reinterpret_cast<const unsigned int *>(src));
    }
}

// All-gather of x by pulling: every rank copies its peers' slices (peer memory, NVLink reads) into
// its own full-length vector.  One launch moves all slices.  The bulk of every slice travels as TMA
// bulk copies driven by ONE thread per CTA — peer memory -> shared-memory ring -> local vector
// (cp.async.bulk + mbarrier; bulk groups for the stores): an NVLink read takes ~3 us, so the link
// only fills with megabytes in flight, which a ring of 16 KB chunks holds without a register
// (profiles/r2_nvlink_copy.txt: 32 such threads reach the copy engines' rate; 128-bit loads need
// every SM for less).  Slices whose ends are not 16-byte aligned, and tails, go element by element.
struct PullSlices {
    const unsigned char *src[SPL_MAX_PEERS];
    unsigned long long dst_off[SPL_MAX_PEERS];     // byte offset of slice g in the full vector
    unsigned long long bytes[SPL_MAX_PEERS];
    int world, rank;
    unsigned int vsize;
};

constexpr uint32_t PULL_CHUNK = 16384;
constexpr int PULL_STAGES = 6, PULL_AHEAD = 4;     // loads run 4 chunks in front of the stores (STAGES >= AHEAD + 2)
constexpr int PULL_THREADS = 128;

__global__ void __launch_bounds__(PULL_THREADS) peer_pull_kernel(PullSlices ps, unsigned char *__restrict__ dst) {
    extern __shared__ __align__(128) unsigned char pull_ring[];
    __shared__ __align__(8) uint64_t full[PULL_STAGES];
    // bulk part of slice k (peers in ring order): whole 16-byte units when both ends are aligned
    unsigned long long b16[SPL_MAX_PEERS], per[SPL_MAX_PEERS];
    const unsigned char *src[SPL_MAX_PEERS];
    unsigned char *out[SPL_MAX_PEERS];
    int np = 0;
    unsigned long long most = 0;
    for (int k = 1; k < ps.world; ++k) {
        const int g = (ps.rank + k) % ps.world;
        src[np] = ps.src[g];
        out[np] = dst + ps.dst_off[g];
        const bool wide = ((((unsigned long long)(uintptr_t)src[np]) | ((unsigned long long)(uintptr_t)out[np])) & 15ull) == 0;
        b16[np] = wide ? ps.bytes[g] & ~15ull : 0ull;
        per[np] = (b16[np] + PULL_CHUNK - 1) / PULL_CHUNK;
        most = per[np] > most ? per[np] : most;
        // what the bulk copies leave: this CTA's share, value by value (all threads but the first), four in flight
        const unsigned long long e0 = b16[np] / ps.vsize, n = ps.bytes[g] / ps.vsize, rest = n - e0;
        if (rest && threadIdx.x > 0) {
            const unsigned long long share = (rest + gridDim.x - 1) / gridDim.x, lo = e0 + blockIdx.x * share,
                                     hi = lo + share < n ? lo + share : n;
            constexpr unsigned long long W = PULL_THREADS - 1;
            auto copy = [&](auto tag) {
                using V = decltype(tag);
                const V *se = reinterpret_cast<const V *>(src[np]);
                V *de = reinterpret_cast<V *>(out[np]);
                unsigned long long e = lo + threadIdx.x - 1;
                for (; e + 3 * W < hi; e += 4 * W) {
                    const V a = __ldcg(se + e), b = __ldcg(se + e + W), c = __ldcg(se + e + 2 * W), d = __ldcg(se + e + 3 * W);
                    de[e] = a; de[e + W] = b; de[e + 2 * W] = c; de[e + 3 * W] = d;
                }
                for (; e < hi; e += W) de[e] = __ldcg(se + e);
            };
            if (ps.vsize == 8) copy((unsigned long long)0);
            else copy((unsigned int)0);
        }
        ++np;
    }
    if (threadIdx.x != 0 || np == 0) return;
    for (int s = 0; s < PULL_STAGES; ++s) mbar_init(full + s, 1);
    mbar_init_fence();
    // chunk id c = j * np + k: chunk j of peer k, so all peers (all links) move at once; ids past a short slice are skipped
    const unsigned long long total = most * np;
    auto locate = [&](unsigned long long c, int &k, unsigned long long &off, uint32_t &len) {
        k = (int)(c % np);
        const unsigned long long j = c / np;
        off = j * PULL_CHUNK;
        len = j < per[k] ? (uint32_t)(b16[k] - off < PULL_CHUNK ? b16[k] - off : PULL_CHUNK) : 0u;
    };
    unsigned long long issued = 0, stored = 0;       // chunks of this CTA that were loaded / stored (skipping empty ids)
    unsigned long long cl = blockIdx.x, cs = blockIdx.x;
    for (;;) {
        // next non-empty chunk to load
        int k; unsigned long long off; uint32_t len = 0;
        while (cl < total) { locate(cl, k, off, len); if (len) break; cl += gridDim.x; }
        const bool more = cl < total;
        if (more) {
            const int s = (int)(issued % PULL_STAGES);
            mbar_expect_tx(full + s, len);
            tma_bulk_g2s(pull_ring + (size_t)s * PULL_CHUNK, src[k] + off, len, full + s);
            ++issued;
            cl += gridDim.x;
        }
        if (issued - stored > (unsigned long long)PULL_AHEAD || (!more && stored < issued)) {
            int k2; unsigned long long off2; uint32_t len2 = 0;
            for (;; cs += gridDim.x) { locate(cs, k2, off2, len2); if (len2) break; }
            const int s = (int)(stored % PULL_STAGES);
            const uint32_t parity = (uint32_t)((stored / PULL_STAGES) & 1);
            mbar_wait(full + s, parity);
            tma_bulk_s2g(out[k2] + off2, pull_ring + (size_t)s * PULL_CHUNK, len2);
            bulk_commit();
            bulk_wait_read_but_one();                   // every store but the newest has left its slot
            ++stored;
            cs += gridDim.x;
        } else if (!more) {
            break;
        }
    }
    bulk_wait_all();
}

// The exchange of the row-sharded transposed product y = A^T x.  Rank g's partial A_g^T x_g covers its footprint
// window [lo_g, hi_g) (spl_spmv_transpose_window) and stays in g's memory; each rank then reads, for every column
// of its own slice of y, the partials of the ranks whose window holds it and folds them in ascending rank: the
// first one copied (a lone -0.0 stays -0.0), the others added; a column no window holds is +0.0.  So y does not
// depend on the ranks' timing.  A banded shard reads its own partial plus two thin halo pieces; a random one the
// world - 1 peers' pieces of its slice.  Every thread keeps RW_COLS columns in flight (coalesced across the warp,
// L2-coherent loads: the peers' partials are read over NVLink).  With flag blocks the flag barrier comes first,
// in every CTA (the arrival stores the same epoch, so repeating it is harmless, and no CTA depends on another
// being resident); a CTA whose wait timed out, or that finds the timeout flag set, writes NaN.
struct ReduceWindows {
    const unsigned char *part[SPL_MAX_PEERS];
    unsigned long long lo[SPL_MAX_PEERS], hi[SPL_MAX_PEERS];
    unsigned long long my0, n;
    int world;
};

constexpr int RW_COLS = 4;
constexpr int RW_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(RW_THREADS)
peer_reduce_windows_kernel(FlagBlocks f, bool barrier, int rank, uint32_t epoch, uint64_t timeout_ns, uint32_t *timed_out,
                           ReduceWindows w, T *__restrict__ y) {
    __shared__ int s_failed;
    bool poison = false;
    if (barrier) {
        if (threadIdx.x == 0) s_failed = 0;
        __syncthreads();
        const int g = threadIdx.x;
        if (g < w.world && g != rank) {
            flag_arrive(f.block[g], rank, epoch);
            if (!flag_wait(f.block[rank] + g, epoch, timeout_ns, 200, timed_out)) s_failed = 1;
        }
        __syncthreads();
        poison = s_failed || *reinterpret_cast<const volatile uint32_t *>(timed_out) != 0u;
    }
    const unsigned long long step = (unsigned long long)gridDim.x * RW_THREADS * RW_COLS;
    for (unsigned long long i0 = (unsigned long long)blockIdx.x * RW_THREADS * RW_COLS + threadIdx.x; i0 < w.n; i0 += step) {
        T acc[RW_COLS];
        bool any[RW_COLS];
#pragma unroll
        for (int u = 0; u < RW_COLS; ++u) { acc[u] = (T)0; any[u] = false; }
#pragma unroll
        for (int g = 0; g < SPL_MAX_PEERS; ++g) {
            if (g >= w.world) break;
            const T *p = reinterpret_cast<const T *>(w.part[g]);
            T v[RW_COLS];
            bool in[RW_COLS];
#pragma unroll
            for (int u = 0; u < RW_COLS; ++u) {
                const unsigned long long c = w.my0 + i0 + (unsigned long long)u * RW_THREADS;
                in[u] = i0 + (unsigned long long)u * RW_THREADS < w.n && c >= w.lo[g] && c < w.hi[g];
                if (in[u]) v[u] = __ldcg(p + (c - w.lo[g]));
            }
#pragma unroll
            for (int u = 0; u < RW_COLS; ++u)
                if (in[u]) { acc[u] = any[u] ? acc[u] + v[u] : v[u]; any[u] = true; }
        }
#pragma unroll
        for (int u = 0; u < RW_COLS; ++u) {
            const unsigned long long i = i0 + (unsigned long long)u * RW_THREADS;
            if (i < w.n) y[i] = poison ? (T)NAN : acc[u];
        }
    }
}

}  // namespace

void peer_reduce_windows(spl_ctx *ctx, int dtype, int world, int rank, const uint64_t *col_starts,
                         const uint64_t *windows, const void *const *partials, void *const *flag_ptrs, uint32_t epoch,
                         uint32_t timeout_ms, void *y_local) {
    FlagBlocks f{};
    ReduceWindows w{};
    w.world = world;
    w.my0 = col_starts[rank];
    w.n = col_starts[rank + 1] - col_starts[rank];
    for (int g = 0; g < world; ++g) {
        w.part[g] = static_cast<const unsigned char *>(partials[g]);
        w.lo[g] = windows[2 * g];
        w.hi[g] = windows[2 * g + 1];
        if (flag_ptrs) f.block[g] = static_cast<uint32_t *>(flag_ptrs[g]);
    }
    const bool barrier = flag_ptrs != nullptr && world > 1;
    const unsigned grid = std::max(1u, std::min(div_up(w.n, (uint64_t)RW_THREADS * RW_COLS), (unsigned)ctx->num_sms * 4u));
    const uint64_t timeout_ns = (uint64_t)(timeout_ms ? timeout_ms : 2000) * 1000000ull;
    if (dtype == SPL_F32)
        peer_reduce_windows_kernel<float><<<grid, RW_THREADS, 0, ctx->stream>>>(f, barrier, rank, epoch, timeout_ns,
                                                                               ctx->d_scratch + 32, w, (float *)y_local);
    else
        peer_reduce_windows_kernel<double><<<grid, RW_THREADS, 0, ctx->stream>>>(f, barrier, rank, epoch, timeout_ns,
                                                                                ctx->d_scratch + 32, w, (double *)y_local);
    check_launch(ctx, "peer_reduce_windows");
}

void peer_pull(spl_ctx *ctx, int world, int rank, size_t vsize, const uint64_t *starts,
               const void *const *slices, void *x_full) {
    SPL_REQUIRE(world >= 1 && world <= SPL_MAX_PEERS && rank >= 0 && rank < world, SPL_ERR_ARG,
                "world must be 1..8 and rank inside it");
    if (world == 1) return;
    PullSlices ps{};
    ps.world = world;
    ps.rank = rank;
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(starts[g] <= starts[g + 1], SPL_ERR_ARG, "starts must be non-decreasing");
        SPL_REQUIRE(slices[g] || starts[g] == starts[g + 1], SPL_ERR_ARG, "NULL slice");
        ps.src[g] = static_cast<const unsigned char *>(slices[g]);
        ps.dst_off[g] = starts[g] * vsize;
        ps.bytes[g] = (starts[g + 1] - starts[g]) * vsize;
    }
    ps.vsize = (unsigned int)vsize;
    const size_t smem = (size_t)PULL_CHUNK * PULL_STAGES;
    SPL_CUDA(cudaFuncSetAttribute(peer_pull_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const char *pc = std::getenv("SPL_PULL_CTAS");                   // measurement knob
    const unsigned ctas = pc ? (unsigned)std::max(1, std::atoi(pc)) : 64u;
    peer_pull_kernel<<<ctas, PULL_THREADS, smem, ctx->stream>>>(ps, static_cast<unsigned char *>(x_full));
    check_launch(ctx, "peer_pull");
}

void peer_barrier_halo(spl_ctx *ctx, int world, int rank, void *const *flag_ptrs, uint32_t epoch, uint32_t timeout_ms,
                       size_t vsize, const uint64_t *starts, void *const *slices, uint32_t halo_left, uint32_t halo_right) {
    SPL_REQUIRE(world >= 1 && world <= SPL_MAX_PEERS && rank >= 0 && rank < world, SPL_ERR_ARG,
                "world must be 1..8 and rank inside it");
    FlagBlocks f{};
    HaloSlices h{};
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(flag_ptrs[g], SPL_ERR_ARG, "NULL flag block");
        SPL_REQUIRE(slices[g] || starts[g] == starts[g + 1], SPL_ERR_ARG, "NULL slice");
        f.block[g] = static_cast<uint32_t *>(flag_ptrs[g]);
        h.slice[g] = static_cast<unsigned char *>(slices[g]);
    }
    for (int g = 0; g <= SPL_MAX_PEERS; ++g) h.start[g] = starts[g < world ? g : world];
    h.halo_left = halo_left;
    h.halo_right = halo_right;
    h.vsize = (unsigned int)vsize;
    peer_barrier_halo_kernel<<<1, 256, 0, ctx->stream>>>(f, world, rank, epoch,
                                                        (uint64_t)(timeout_ms ? timeout_ms : 2000) * 1000000ull,
                                                        ctx->d_scratch + 32, h);
    check_launch(ctx, "peer_barrier_halo");
}

void peer_barrier(spl_ctx *ctx, int world, int rank, void *const *flag_ptrs, uint32_t epoch,
                  uint32_t timeout_ms) {
    SPL_REQUIRE(world >= 1 && world <= SPL_MAX_PEERS && rank >= 0 && rank < world, SPL_ERR_ARG,
                "world must be 1..8 and rank inside it");
    if (world == 1) return;
    FlagBlocks f{};
    for (int g = 0; g < world; ++g) {
        SPL_REQUIRE(flag_ptrs[g], SPL_ERR_ARG, "NULL flag block");
        f.block[g] = static_cast<uint32_t *>(flag_ptrs[g]);
    }
    peer_barrier_kernel<<<1, 32, 0, ctx->stream>>>(f, world, rank, epoch,
                                                   (uint64_t)(timeout_ms ? timeout_ms : 2000) * 1000000ull,
                                                   ctx->d_scratch + 32);
    check_launch(ctx, "peer_barrier");
}

}  // namespace spl
