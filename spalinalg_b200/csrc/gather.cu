// gather.cu — row-sharded y = A x for GENERAL shards (random / unstructured columns), the
// all-gather of x fused into the product (SURVEY.md 8e, "Collective (general)").
//
// A banded or stencil shard copies its few halo columns inside the barrier kernel (peer.cu).  A
// shard with random columns cannot: every remote gather would be a 4-byte NVLink transaction.  It
// needs the whole of x locally, and done as "all-gather, then SpMV" the exchange (35 MB per rank at
// 8 GPUs on config 3) costs as much as the product and nothing overlaps.  Here ONE persistent
// kernel does both:
//   * the shard is stored blocked by column owner: block 0 holds, row by row, the entries whose
//     column lives on this rank, the following blocks the peers' columns in ring order (rank+1,
//     rank+2, ...), one block per peer or per GROUP of consecutive peers (block_first);
//   * every CTA carries one COPY warp beside its 8 compute warps.  Its elected thread moves the
//     CTA's share of the peers' slices with TMA bulk copies: peer memory -> a small shared-memory
//     ring -> the local full-length x (cp.async.bulk + mbarrier, bulk groups for the stores), three
//     2 KB loads in flight per CTA = several MB in flight on the chip, which is what a ~3 us NVLink
//     round trip needs (profiles/r2_nvlink_copy.txt: 128-bit loads from 64 CTAs reach 400 GB/s
//     alone and 220 GB/s beside the gathers of the product, which saturate the same L1/LSU path;
//     TMA bypasses it and reaches the copy engines' rate with one thread per CTA).  When a CTA's
//     chunks of a slice have been written it bumps that slice's counter (release);
//   * the COMPUTE warps own a fixed range of rows per CTA, keep the row sums in shared memory, and
//     walk the blocks in order: block 0 needs only the rank's own slice and runs while the first
//     slices are in flight; before block b they wait (acquire) for the counters of its slices.
//     Transfer and math overlap block by block, and y is written once.  A tile producer warp feeds
//     them the tiles of the stream kernel (stream_tile.cuh: same tile, same row loop, same bits per
//     block); the copies and the folded flag barrier use the primitives of ptx.cuh.
// All CTAs are resident at once (cooperative launch: the grid is what fits), so the waits cannot
// deadlock.  Row sums add the blocks in ring order, not in ascending column order: tolerance parity
// (1e-12 / 1e-5), like every multi-lane kernel.
#include <algorithm>
#include <cstdlib>

#include "kernels.cuh"
#include "ptx.cuh"
#include "stream_tile.cuh"

namespace spl {

namespace {

struct GatherPeers {
    const void *slice[SPL_MAX_PEERS];
    uint32_t start[SPL_MAX_PEERS + 1];
    int world, rank;
};

// The device-side barrier of spl_peer_barrier, folded into the kernel: flags[g] = rank g's flag block
// (peer memory), flags_mine = this rank's own block (NULL: the caller ran the barrier itself)
struct GatherBarrier {
    uint32_t *flags[SPL_MAX_PEERS];
    const uint32_t *flags_mine;
    uint32_t epoch;
    unsigned long long timeout_ns;
    uint32_t *failed;
};

constexpr int GF_CTA = TILE_CONSUMERS + 64;      // the consumers, one warp that feeds them tiles, one that copies x
constexpr uint32_t GF_CHUNK = 4096;      // bytes per bulk copy of x: 5 x 4 KB in flight per CTA, ~9 MB on the chip — beside the
                                         // product's gathers an NVLink read takes ~15 us, and 4 MB in flight gave 240 GB/s
constexpr int GF_STAGES = 6;             // x ring slots per CTA
constexpr int GF_AHEAD = 4;              // loads run this many chunks in front of the stores (STAGES >= AHEAD + 2)
constexpr uint32_t GF_RING = GF_CHUNK * GF_STAGES;

// block b of the shard = the columns owned by ring offsets [first[b], first[b+1]); first[0] = 0, first[1] = 1
struct GatherBlocks {
    uint32_t first[SPL_MAX_PEERS + 1];
    int n;
};

// ---- the copy warp of one CTA ----
template <typename T>
__device__ void gather_copy_warp(const GatherPeers &gp, T *x_full, uint32_t *ready, const GatherBarrier &gb,
                                 unsigned char *ring, uint64_t *full, unsigned long long *timeline) {
    const int G = gp.world;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned long long cta = blockIdx.x, ncta = gridDim.x;
    if (gb.flags_mine) {
        // fused barrier, arrival: this rank's published slice is final (stream order put its writers before us)
        if (cta == 0 && (int)lane < G && (int)lane != gp.rank) flag_arrive(gb.flags[lane], gp.rank, gb.epoch);
        __syncwarp();
    }
    // fused barrier, wait: rank g's slice is final once its epoch shows up in this rank's flag block; waited for
    // slice by slice, so a late peer delays only its own slice
    auto wait_owner = [&](int g) {
        if (gb.flags_mine) flag_wait(gb.flags_mine + g, gb.epoch, gb.timeout_ns, 100, gb.failed);
    };
    // chunks of the bulk path per slice (ring offset k = 1..G-1): whole 16-byte units of slices whose two ends are
    // 16-byte aligned (IPC blocks are; slice starts of an f32 vector need not be); the rest goes element by element
    unsigned long long cum[SPL_MAX_PEERS + 1];             // cum[k] = chunks in ring offsets 1..k
    cum[0] = 0;
    for (int k = 1; k < G; ++k) {
        const int g = (gp.rank + k) % G;
        const unsigned char *src = static_cast<const unsigned char *>(gp.slice[g]);
        unsigned char *dst = reinterpret_cast<unsigned char *>(x_full + gp.start[g]);
        const unsigned long long n = gp.start[g + 1] - gp.start[g], bytes = n * sizeof(T);
        const bool wide = ((((unsigned long long)(uintptr_t)src) | ((unsigned long long)(uintptr_t)dst)) & 15ull) == 0;
        const unsigned long long b16 = wide ? bytes & ~15ull : 0ull;
        cum[k] = cum[k - 1] + (b16 + GF_CHUNK - 1) / GF_CHUNK;
        // elements outside the bulk path: this CTA's share, all lanes
        const unsigned long long e0 = b16 / sizeof(T), rest = n - e0;
        if (rest) {
            if (lane == 0) wait_owner(g);
            __syncwarp();
            const T *se = reinterpret_cast<const T *>(src);
            T *de = reinterpret_cast<T *>(dst);
            const unsigned long long per = (rest + ncta - 1) / ncta, lo = e0 + cta * per,
                                     hi = lo + per < n ? lo + per : n;
            for (unsigned long long e = lo + lane; e < hi; e += 32) de[e] = __ldcg(se + e);
        }
    }
    __syncwarp();
    if (lane == 0) {
        for (int s = 0; s < GF_STAGES; ++s) mbar_init(full + s, 1);
        mbar_init_fence();
        const unsigned long long total = cum[G - 1];
        const unsigned long long mine = total > cta ? (total - cta + ncta - 1) / ncta : 0;
        int kl = 1, ks = 1, ksig = 1, kw = 0;
        __threadfence();                                                               // the warp's element-path stores above
        for (; ksig < G && cum[ksig] <= cta; ++ksig) atomicAdd(ready + ksig, 1u);      // slices that hold no chunk of this CTA
        auto slice_of = [&](int k, const unsigned char *&src, unsigned char *&dst, unsigned long long &b16) {
            const int g = (gp.rank + k) % G;
            src = static_cast<const unsigned char *>(gp.slice[g]);
            dst = reinterpret_cast<unsigned char *>(x_full + gp.start[g]);
            b16 = ((unsigned long long)(gp.start[g + 1] - gp.start[g]) * sizeof(T)) & ~15ull;
        };
        for (unsigned long long i = 0; i < mine + GF_AHEAD; ++i) {
            if (i < mine) {
                const unsigned long long c = cta + i * ncta;
                while (c >= cum[kl]) ++kl;
                for (; kw < kl; ++kw) {                                          // owners of the slices up to kl have arrived
                    wait_owner((gp.rank + kw + 1) % G);
                    if (timeline && cta == 0 && kw == 0) timeline[0] = global_timer_ns();
                }
                const unsigned char *src; unsigned char *dst; unsigned long long b16;
                slice_of(kl, src, dst, b16);
                const unsigned long long off = (c - cum[kl - 1]) * GF_CHUNK;
                const uint32_t len = (uint32_t)(b16 - off < GF_CHUNK ? b16 - off : GF_CHUNK);
                const int s = (int)(i % GF_STAGES);
                mbar_expect_tx(full + s, len);
                tma_bulk_g2s(ring + (size_t)s * GF_CHUNK, src + off, len, full + s);
            }
            if (i >= (unsigned long long)GF_AHEAD) {
                const unsigned long long j = i - GF_AHEAD, c = cta + j * ncta;
                while (c >= cum[ks]) ++ks;
                const unsigned char *src; unsigned char *dst; unsigned long long b16;
                slice_of(ks, src, dst, b16);
                const unsigned long long off = (c - cum[ks - 1]) * GF_CHUNK;
                const uint32_t len = (uint32_t)(b16 - off < GF_CHUNK ? b16 - off : GF_CHUNK);
                const int s = (int)(j % GF_STAGES);
                const uint32_t parity = (uint32_t)((j / GF_STAGES) & 1);
                mbar_wait(full + s, parity);
                tma_bulk_s2g(dst + off, ring + (size_t)s * GF_CHUNK, len);
                bulk_commit();
                if (c + ncta >= cum[ks]) {
                    // this CTA's last chunk of the slice: wait until its stores are WRITTEN (the loads ahead keep flying —
                    // bulk groups count stores only), then say so.  Slices that lie wholly below the next chunk hold
                    // nothing of this CTA that is still in flight
                    bulk_wait_all();
                    __threadfence();
                    for (; ksig < G && cum[ksig] <= c + ncta; ++ksig) atomicAdd(ready + ksig, 1u);
                } else {
                    bulk_wait_read_but_one();            // every store but the newest has left its slot
                }
            }
        }
        bulk_wait_all();
        __threadfence();
        for (; ksig < G; ++ksig) atomicAdd(ready + ksig, 1u);
    }
}

// Shared memory of a CTA: [tile stages: indices | values | row pointers] [x ring] [tile bounds] [barriers]
struct GatherShape {
    uint32_t rows_per_cta;    // multiple of 32
    uint32_t ntiles;          // tiles of R rows per block and CTA
    uint32_t cap;             // entries a tile stage holds (16-byte aligned superset of the largest tile)
    uint32_t stages;          // tile stages
    uint32_t off_val, off_ptr, off_ring, off_tlo, off_bar;      // byte offsets
};

template <typename T, int LPR, int U>
__global__ void __launch_bounds__(GF_CTA, 4)
spmv_gather_fused_kernel(uint32_t nloc, const uint32_t *__restrict__ bptr, uint32_t pstride,
                         const uint32_t *__restrict__ bind, const T *__restrict__ bval, GatherPeers gp, GatherBlocks gk,
                         T *x_full, T *__restrict__ y, uint32_t *ready, uint32_t target, GatherShape sh, GatherBarrier gb,
                         unsigned long long *timeline) {
    constexpr uint32_t R = tile_rows(LPR), PTRS = tile_ptr_slots(R);
    extern __shared__ __align__(128) unsigned char gf_raw[];
    uint32_t *s_ind = reinterpret_cast<uint32_t *>(gf_raw);
    T *s_val = reinterpret_cast<T *>(gf_raw + sh.off_val);
    uint32_t *s_ptr = reinterpret_cast<uint32_t *>(gf_raw + sh.off_ptr);
    uint32_t *s_tlo = reinterpret_cast<uint32_t *>(gf_raw + sh.off_tlo);
    uint64_t *full = reinterpret_cast<uint64_t *>(gf_raw + sh.off_bar);
    uint64_t *empty = full + sh.stages;
    uint64_t *xfull = empty + sh.stages;
    const uint32_t c = blockIdx.x;
    const uint64_t rs64 = (uint64_t)c * sh.rows_per_cta;
    const uint32_t rs = rs64 < nloc ? (uint32_t)rs64 : nloc;
    const uint32_t re = rs + sh.rows_per_cta < nloc ? rs + sh.rows_per_cta : nloc;
    const uint32_t ntiles = (re - rs + R - 1) / R;          // 0 for a CTA without rows (it still copies x)
    const uint32_t nb = (uint32_t)gk.n;

    if (threadIdx.x >= TILE_CONSUMERS + 32) {
        // ---- warp 9: this CTA's share of the peers' slices of x ----
        if (gp.world > 1) gather_copy_warp<T>(gp, x_full, ready, gb, gf_raw + sh.off_ring, xfull, timeline);
        return;
    }
    if (threadIdx.x >= TILE_CONSUMERS) {
        // ---- warp 8: feeds the consumers.  All lanes fetch the tile bounds of every block (one round trip), then one
        // thread issues the bulk copies of each tile's row pointers, indices and values, `stages` tiles ahead; the
        // matrix does not depend on x, so the tiles of block b are in shared memory before its slices have landed ----
        const uint32_t lane = threadIdx.x & 31u;
        if (ntiles == 0) return;
        for (uint32_t i = lane; i < nb * (ntiles + 1); i += 32) {
            const uint32_t k = i / (ntiles + 1), t = i % (ntiles + 1);
            const uint32_t r = rs + t * R < re ? rs + t * R : re;
            s_tlo[i] = __ldg(bptr + (size_t)k * pstride + r);
        }
        if (lane == 0) {
            for (uint32_t s = 0; s < sh.stages; ++s) {
                mbar_init(full + s, 1);
                mbar_init(empty + s, TILE_CONSUMERS / 32);
            }
            mbar_init_fence();
        }
        __syncwarp();
        asm volatile("bar.arrive 2, %0;" ::"n"(TILE_CONSUMERS + 32) : "memory");      // barriers are live: consumers may wait on them
        if (lane != 0) return;
        const uint64_t pol = l2_policy_evict_first();
        uint32_t s = 0, phase = 0, i = 0;
        for (uint32_t k = 0; k < nb; ++k)
            for (uint32_t t = 0; t < ntiles; ++t, ++i) {
                const uint32_t lo = s_tlo[k * (ntiles + 1) + t], hi = s_tlo[k * (ntiles + 1) + t + 1];
                if (i >= sh.stages) mbar_wait(empty + s, phase ^ 1u);
                const uint32_t za = slice_lo(lo);
                uint32_t cnt = slice_hi(hi) - za;
                if (cnt > sh.cap) {                        // tile_entries_max was too small: never overrun the stage — the
                    atomicExch(gb.failed, 1u);             // tile is cut (the consumers clamp too) and y comes back as NaN
                    cnt = sh.cap;
                }
                const uint32_t r0 = rs + t * R;
                const uint32_t left = (pstride - r0) & ~3u;                   // pointer entries from r0 to the end of the block's array
                const uint32_t np = left < PTRS ? left : PTRS;
                mbar_expect_tx(full + s, cnt * (uint32_t)(sizeof(uint32_t) + sizeof(T)) + np * (uint32_t)sizeof(uint32_t));
                tma_bulk_g2s(s_ptr + (size_t)s * PTRS, bptr + (size_t)k * pstride + r0, np * (uint32_t)sizeof(uint32_t), full + s);
                if (cnt) {
                    tma_bulk_g2s_hint(s_ind + (size_t)s * sh.cap, bind + za, cnt * (uint32_t)sizeof(uint32_t), full + s, pol);
                    tma_bulk_g2s_hint(s_val + (size_t)s * sh.cap, bval + za, cnt * (uint32_t)sizeof(T), full + s, pol);
                }
                if (++s == sh.stages) { s = 0; phase ^= 1u; }
            }
        return;
    }

    // ---- consumers: LPR lanes per row (tile_row_sum) — pointers, indices and values come from shared memory, only x
    // from global memory, and the warps run on their own (no CTA barrier).
    // A row's running sum lives in y itself: the same lanes own the row in every block, and shared memory spent on
    // sums would come out of the L1 that holds the gathers in flight.  Measured alternatives (entries dealt to the
    // lanes with eight gathers each, four rows per lane, products summed in a second pass) kept more gathers in flight
    // and were all slower: profiles/r2_spmv_notes.md ----
    if (ntiles == 0) return;
    asm volatile("bar.sync 2, %0;" ::"n"(TILE_CONSUMERS + 32) : "memory");
    const T *own = static_cast<const T *>(gp.slice[gp.rank]) - gp.start[gp.rank];
    const uint32_t lane = threadIdx.x & 31u, rl = threadIdx.x / LPR, sub = threadIdx.x % LPR;
    const bool stamp = timeline && c == 0 && threadIdx.x == 0;
    uint32_t s = 0, phase = 0;
    for (uint32_t k = 0; k < nb; ++k) {
        if (stamp) timeline[1 + 3 * k] = global_timer_ns();                                           // block k: wait begins
        if (k > 0) {
            if (lane == 0)
                for (uint32_t o = gk.first[k]; o < gk.first[k + 1]; ++o)
                    while ((int32_t)(ld_acquire_gpu(ready + o) - target) < 0) __nanosleep(64);
            __syncwarp();
        }
        if (stamp) timeline[2 + 3 * k] = global_timer_ns();                                           // its slices have landed
        for (uint32_t t = 0; t < ntiles; ++t) {
            mbar_wait(full + s, phase);
            const uint32_t *cp = s_ptr + (size_t)s * PTRS;
            const uint32_t *ci = s_ind + (size_t)s * sh.cap;
            const T *cv = s_val + (size_t)s * sh.cap;
            const uint32_t r = rs + t * R + rl;
            const uint32_t za = slice_lo(cp[0]);
            uint32_t p0 = 0, e = 0;
            if (r < re) { p0 = min(cp[rl] - za, sh.cap); e = min(cp[rl + 1] - za, sh.cap); }      // never past the stage
            T prev = (T)0;
            if (k > 0 && sub == 0 && r < re) prev = y[r];              // in flight with the gathers
            T acc = (T)0;
            // block 0 reads the published slice (constant for the whole kernel); x_full is written by this very kernel,
            // behind the acquire that let this block start: L2 loads
            if (k == 0) tile_row_sum<T, LPR, U>(acc, ci, 0, cv, p0, e, sub, [&](uint32_t col) { return __ldg(own + col); });
            else tile_row_sum<T, LPR, U>(acc, ci, 0, cv, p0, e, sub, [&](uint32_t col) { return __ldcg(x_full + col); });
            __syncwarp();
            if (lane == 0) mbar_arrive(empty + s);
            acc = row_lanes_sum<LPR>(acc);
            if (sub == 0 && r < re) y[r] = prev + acc;
            if (++s == sh.stages) { s = 0; phase ^= 1u; }
        }
        if (stamp) timeline[3 + 3 * k] = global_timer_ns();                                           // block k done (this warp)
    }
    // a fused barrier that gave up: NaN instead of sums over a half-written x (the status call reports it)
    const bool poisoned = gb.failed && *reinterpret_cast<const volatile uint32_t *>(gb.failed) != 0u;
    if (poisoned && sub == 0)
        for (uint32_t t = 0; t < ntiles; ++t) {                          // every lane poisons the rows it summed
            const uint32_t r = rs + t * R + rl;
            if (r < re) y[r] = (T)NAN;
        }
    if (timeline && threadIdx.x == 0) atomicMax(timeline + 1 + 3 * nb, global_timer_ns());           // the last CTA to finish
}

}  // namespace

// Launch shape: three CTAs per SM (cooperative launch: all resident), two or three tile stages, within `smem_per_sm`
// bytes of shared memory per SM.  The budget matters: what the kernel does not take stays L1, and L1 lines are where
// the gathers in flight land — with 200 KB of staging the same gathers ran three times slower (profiles/
// r2_spmv_notes.md).  Returns false when the tile does not fit the budget.  tile_caps = the most entries any 64 / 128 /
// 256 / 512 / 1024 consecutive rows (starting at a multiple of 32) hold in one block.
template <typename T, int LPR, int U>
bool spmv_gather_fused_t(size_t smem_per_sm, spl_ctx *ctx, uint32_t nloc, const uint32_t *bptr, uint32_t pstride, const uint32_t *bind,
                         const T *bval, const uint32_t *tile_caps, const GatherPeers &gp, const GatherBlocks &gk, T *x_full,
                         T *y, uint32_t *ready, uint32_t epoch, const GatherBarrier &gb, unsigned long long *timeline) {
    auto k = spmv_gather_fused_kernel<T, LPR, U>;
    constexpr uint32_t R = tile_rows(LPR);
    static_assert(R == 64 || R == 128 || R == 256, "tile rows");
    const uint32_t cap = stage_capacity(tile_caps[R == 64 ? 0 : R == 128 ? 1 : 2]);
    const char *pc = std::getenv("SPL_GATHER_CTAS_PER_SM");          // measurement knobs
    const char *ps = std::getenv("SPL_GATHER_STAGES");
    const int most = pc ? std::max(1, std::atoi(pc)) : 3;
    uint32_t ncta = 0;
    size_t smem = 0;
    GatherShape sh{};
    auto shape = [&](uint32_t ctas, uint32_t stages) {
        sh.rows_per_cta = (uint32_t)(((uint64_t)nloc + ctas - 1) / ctas);
        sh.rows_per_cta = (sh.rows_per_cta + 31u) & ~31u;
        sh.ntiles = (sh.rows_per_cta + R - 1) / R;
        sh.cap = cap;
        sh.stages = stages;
        size_t o = (size_t)stages * cap * sizeof(uint32_t);
        sh.off_val = (uint32_t)o;
        o += (size_t)stages * cap * sizeof(T);
        sh.off_ptr = (uint32_t)o;
        o += (size_t)stages * tile_ptr_slots(R) * sizeof(uint32_t);
        o = (o + 127) & ~(size_t)127;
        sh.off_ring = (uint32_t)o;
        o += GF_RING;
        sh.off_tlo = (uint32_t)o;
        o += (size_t)gk.n * (sh.ntiles + 1) * sizeof(uint32_t);
        o = (o + 7) & ~(size_t)7;
        sh.off_bar = (uint32_t)o;
        o += (size_t)(2 * stages + GF_STAGES) * sizeof(uint64_t);
        return o;
    };
    for (int want = most; want >= 1 && ncta == 0; --want)
        // two tile stages by default: a third measured 3 % faster on 8 GPUs (1.25 M rows per rank) and 36 % SLOWER on
        // 2 GPUs (5 M rows per rank: 0.62 against 0.39 ms, profiles/r2_bench_n2.json); what it costs is L1
        for (uint32_t stages = ps ? (uint32_t)std::max(2, std::atoi(ps)) : 2u; stages >= 2 && ncta == 0; --stages) {
            const uint32_t ctas = (uint32_t)ctx->num_sms * (uint32_t)want;
            smem = shape(ctas, stages);
            if (smem > smem_per_sm / (size_t)want) continue;
            if (smem > 48 * 1024) SPL_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int resident = 0;
            SPL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, k, GF_CTA, smem));
            if (resident >= want) ncta = ctas;
        }
    if (ncta == 0) return false;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(ncta);
    cfg.blockDim = dim3(GF_CTA);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;           // all CTAs resident or the launch fails: the waits cannot hang
    at[0].val.cooperative = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    SPL_CUDA(cudaLaunchKernelEx(&cfg, k, nloc, bptr, pstride, bind, bval, gp, gk, x_full, y, ready, epoch * ncta, sh, gb,
                                timeline));
    check_launch(ctx, "spmv_gather_fused");
    return true;
}

void spmv_gather_fused(spl_ctx *ctx, int dtype, uint32_t nloc, int world, int rank, const uint64_t *col_starts,
                       const void *const *x_slices, int nblocks, const uint32_t *block_first, const uint32_t *bptr,
                       uint32_t pstride, const uint32_t *tile_caps, const uint32_t *bind, const void *bval, void *x_full,
                       void *y, uint32_t *ready, uint32_t epoch, double entries_per_row, void *const *flag_ptrs,
                       uint32_t barrier_epoch, uint32_t timeout_ms, unsigned long long *timeline) {
    GatherBarrier gb{};
    if (flag_ptrs && world > 1) {
        for (int g = 0; g < world; ++g) gb.flags[g] = static_cast<uint32_t *>(flag_ptrs[g]);
        gb.flags_mine = gb.flags[rank];
        gb.epoch = barrier_epoch;
        gb.timeout_ns = (unsigned long long)(timeout_ms ? timeout_ms : 2000) * 1000000ull;
    }
    gb.failed = ctx->d_scratch + 32;
    GatherPeers gp{};
    gp.world = world;
    gp.rank = rank;
    for (int g = 0; g <= SPL_MAX_PEERS; ++g) gp.start[g] = (uint32_t)col_starts[g < world ? g : world];
    for (int g = 0; g < world; ++g) gp.slice[g] = x_slices[g];
    GatherBlocks gk{};
    uint32_t widest = 1;
    if (block_first) {
        SPL_REQUIRE(nblocks >= 1 && nblocks <= world && block_first[0] == 0 && block_first[nblocks] == (uint32_t)world &&
                        (world == 1 || block_first[1] == 1),
                    SPL_ERR_ARG, "block_first must run 0, 1, ..., world (block 0 = the own slice alone)");
        gk.n = nblocks;
        for (int b = 0; b <= nblocks; ++b) gk.first[b] = block_first[b];
        for (int b = 0; b < nblocks; ++b) {
            SPL_REQUIRE(block_first[b] < block_first[b + 1], SPL_ERR_ARG, "block_first must increase");
            widest = std::max(widest, block_first[b + 1] - block_first[b]);
        }
    } else {
        gk.n = world;
        for (int b = 0; b <= world; ++b) gk.first[b] = (uint32_t)b;
    }
    // entries a row holds in the WIDEST block
    const double e = entries_per_row * (double)widest / (double)world;
    auto go = [&](auto tag, auto lpr, auto u, size_t smem_per_sm) {
        using T = decltype(tag);
        return spmv_gather_fused_t<T, decltype(lpr)::value, decltype(u)::value>(smem_per_sm, ctx, nloc, bptr, pstride, bind,
                                                                               (const T *)bval, tile_caps, gp, gk, (T *)x_full,
                                                                               (T *)y, ready, epoch, gb, timeline);
    };
    using I1 = std::integral_constant<int, 1>;
    using I2 = std::integral_constant<int, 2>;
    using I4 = std::integral_constant<int, 4>;
    // lanes per row from the entries a row holds in the widest block; more lanes (a smaller tile) when the tile does
    // not fit the shared-memory budget; as a last resort any tile that fits the SM at all
    const char *pl = std::getenv("SPL_GATHER_LANES");                // measurement knobs
    const char *pk = std::getenv("SPL_GATHER_SMEM_KB");
    const size_t budget = (size_t)(pk ? std::max(16, std::atoi(pk)) : 128) * 1024;
    const int lanes = pl ? std::atoi(pl) : (e <= 4.0 ? 1 : e <= 16.0 ? 2 : 4);
    auto pick = [&](auto tag) {
        for (size_t limit : {budget, (size_t)226 * 1024}) {
            if (lanes <= 1 && go(tag, I1{}, I4{}, limit)) return;
            if (lanes <= 2 && go(tag, I2{}, I4{}, limit)) return;
            if (go(tag, I4{}, I4{}, limit)) return;
        }
        SPL_REQUIRE(false, SPL_ERR_UNSUPPORTED, "fused gather SpMV: 64 rows of one block of the shard do not fit in shared memory");
    };
    if (dtype == SPL_F32) pick(float{});
    else pick(double{});
}

}  // namespace spl
