// spmv.cu — y = A x for CSR A and dense x, y.
//
// The reference has no SpMV; its pinned meaning is `&A * &X` with X an n x 1 matrix
// (src/csr/ops/mul.rs:5-60): per row the column-ascending sum of round(a*x).  Parity bar
// (BASELINE.json north_star): 1e-12 (f64) / 1e-5 (f32) relative, so the in-row reduction
// order is free.  Three hand-written kernels:
//   vector  LPR lanes per row (1..32) with 4 entries in flight per lane: consecutive lanes read
//           consecutive entries (col/val loads coalesce, neighbouring columns share x-gather
//           sectors), shuffle reduction.  Regular rows (stencils, bands, uniform random).  The x
//           access is a template policy: one local array, or the slice of the rank that owns the
//           column (peer memory over NVLink: the row-sharded product without a collective).
//   split   merge-path's balance at warp granularity: every warp owns a fixed chunk of stored
//           entries, rows are found from a per-chunk start row, rows that straddle chunks go
//           through a deterministic carry fix-up.  Skewed (power-law) rows; with a shared-memory
//           cache of the hottest x values from the second product on a matrix.
//   merge   merge-path tiles over (row ends, nnz): every CTA takes the same number of
//           (row + nnz) items; its contiguous col/val slice arrives in shared memory by TMA bulk
//           copies (cp.async.bulk + mbarrier), products are formed in place, rows are reduced by
//           a balanced per-thread path walk and a segmented shuffle scan; partial rows go to a
//           deterministic fix-up.  Kept selectable; the split kernel replaced it in the planner.
// 128-bit per-lane loads of col/val were measured and rejected for the gather-bound patterns:
// they put entries 4 apart on neighbouring lanes and triple the L1 wavefronts of the x gathers
// (DESIGN.md, "SpMV").
// Algorithmic bytes per launch: nnz*(4+V) + (ncols+nrows)*V  (SURVEY.md 8d); HBM-bound.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "kernels.cuh"
#include "ptx.cuh"
#include "radix_sort.cuh"
#include "scan.cuh"
#include "stream_tile.cuh"

namespace spl {

namespace {

// ------------------------------------------------------------------ vector kernel
// Where x[c] comes from.  XLocal: one device array.  XPeer: the slice of the rank that owns
// column c — this GPU's HBM for the own block, a peer's HBM over NVLink (CUDA IPC mapping)
// otherwise; the exchange of x is the gather itself, there is no staging copy and no collective.
template <typename T>
struct XLocal {
    const T *x;
    __device__ __forceinline__ T operator()(uint32_t c) const { return __ldg(x + c); }
    __device__ __forceinline__ bool poisoned() const { return false; }
    __device__ __forceinline__ bool all_local(uint32_t, uint32_t) const { return true; }
    __device__ __forceinline__ T local(uint32_t c) const { return __ldg(x + c); }
};
template <typename T>
struct XPeer {
    const T *mine;
    uint32_t my_start, my_len;
    const T *slice[SPL_MAX_PEERS];
    uint32_t start[SPL_MAX_PEERS + 1];
    int world;
    const uint32_t *barrier_failed;          // set by a peer barrier that timed out on this context
    // A product behind a barrier that gave up would read a peer's slice before it is final: its rows
    // come out as NaN instead of plausible numbers (the status call reports the timeout itself).
    __device__ __forceinline__ bool poisoned() const { return *reinterpret_cast<const volatile uint32_t *>(barrier_failed) != 0u; }
    __device__ __forceinline__ T operator()(uint32_t c) const {
        const uint32_t o = c - my_start;
        if (o < my_len) return __ldg(mine + o);
        const T *p = mine;                       // never dereferenced at index o: c is in some block
        uint32_t off = 0;
#pragma unroll
        for (int g = 0; g < SPL_MAX_PEERS; ++g)
            if (g < world && c >= start[g] && c < start[g + 1]) { p = slice[g]; off = c - start[g]; }
        return __ldcg(p + off);                  // peer HBM: L2-coherent load, not kept in L1
    }
    // Rows whose columns all lie in the own block (every row but the few at the edges of a banded or
    // stencil shard) take a loop without the owner test: a branch per gather keeps a lane's U gathers
    // from issuing back to back (measured: 0.82 of the HBM peak per rank against 1.02 on one GPU).
    __device__ __forceinline__ bool all_local(uint32_t cmin, uint32_t cmax) const {
        return cmin - my_start < my_len && cmax - my_start < my_len;
    }
    __device__ __forceinline__ T local(uint32_t c) const { return __ldg(mine + (c - my_start)); }
};

template <typename T, int LPR, typename XG>
__global__ void __launch_bounds__(256)
spmv_vector_kernel(uint32_t nrows, const uint32_t *__restrict__ ptr,
                   const uint32_t *__restrict__ ind, const T *__restrict__ val, const XG xg,
                   T *__restrict__ y) {
    constexpr int U = 4;   // entries in flight per lane: all col/val loads, then all x gathers
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t row = gtid / LPR;
    const uint32_t sub = (uint32_t)(gtid % LPR);
    T acc = (T)0;
    if (row < nrows) {
        uint32_t p = __ldg(ptr + row) + sub;
        const uint32_t e = __ldg(ptr + row + 1);
        for (; p < e; p += U * LPR) {
            uint32_t c[U];
            T v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t pu = p + u * LPR;
                const bool ok = pu < e;
                const uint32_t idx = ok ? pu : p;        // p itself is in range: safe dummy
                c[u] = __ldg(ind + idx);     // L1-allocating on purpose: with few lanes per row a warp
                v[u] = __ldg(val + idx);     // touches 32 rows' sectors and re-reads them from L1
            }
            T xv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) xv[u] = xg(c[u]);
#pragma unroll
            for (int u = 0; u < U; ++u) acc += p + u * LPR < e ? v[u] * xv[u] : (T)0;   // 0, never 0 * inf
        }
    }
    acc = row_lanes_sum<LPR>(acc);
    if (sub == 0 && row < nrows) y[row] = xg.poisoned() ? (T)NAN : acc;
}

// rows [r0, r1) of A: y[r0, r1)
template <typename T, int LPR, typename XG>
void launch_vector(spl_ctx *ctx, const spl_mat *a, const XG &xg, T *y, uint32_t r0, uint32_t r1) {
    const uint64_t threads = (uint64_t)(r1 - r0) * LPR;
    spmv_vector_kernel<T, LPR, XG><<<div_up(threads, 256), 256, 0, ctx->stream>>>(
        r1 - r0, a->ptr + r0, a->ind, static_cast<const T *>(a->val), xg, y + r0);
    check_launch(ctx, "spmv_vector");
}

template <typename T, typename XG>
void spmv_vector(spl_ctx *ctx, const spl_mat *a, const XG &xg, T *y, int lanes, uint32_t r0, uint32_t r1) {
    switch (lanes) {
        case 1: launch_vector<T, 1>(ctx, a, xg, y, r0, r1); break;
        case 2: launch_vector<T, 2>(ctx, a, xg, y, r0, r1); break;
        case 4: launch_vector<T, 4>(ctx, a, xg, y, r0, r1); break;
        case 8: launch_vector<T, 8>(ctx, a, xg, y, r0, r1); break;
        case 16: launch_vector<T, 16>(ctx, a, xg, y, r0, r1); break;
        case 32: launch_vector<T, 32>(ctx, a, xg, y, r0, r1); break;
        default: throw Error{SPL_ERR_ARG, "lanes per row must be 1, 2, 4, 8, 16 or 32"};
    }
}

// ------------------------------------------------------------------ sliced kernel
// The vector kernel with more than one lane per row spends its L1 bandwidth on partial sectors (a
// warp's load touches 32/LPR rows, 16-32 useful bytes of each line) and its rows pay a shuffle
// reduction; with one lane per row on CSR the loads of a warp are a stride of one row length apart.
// Regular matrices therefore get a second copy in slices of 32 consecutive rows, stored column-major
// inside the slice and padded to the slice's longest row: lane = row, step k of a warp reads one
// full line of indices and one or two of values, no shuffles, and the sum runs in ascending column
// order — bit-identical to the reference's `&A * &X` (src/csr/ops/mul.rs:25-40).  Padded slots are
// never multiplied (0, never 0 * inf).
__global__ void slice_width_kernel(const uint32_t *__restrict__ ptr, uint32_t nrows, uint32_t nslices,
                                   uint32_t *__restrict__ width) {
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t slice = gtid >> 5;
    if (slice >= nslices) return;
    uint32_t len = gtid < nrows ? ptr[gtid + 1] - ptr[gtid] : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
    if (lane_id() == 0) width[slice] = len;
}

template <typename T>
__global__ void __launch_bounds__(256)
slice_fill_kernel(const uint32_t *__restrict__ ptr, const uint32_t *__restrict__ ind, const T *__restrict__ val,
                  uint32_t nrows, uint32_t nslices, const uint32_t *__restrict__ slice_ptr,
                  uint32_t *__restrict__ slice_ind, T *__restrict__ slice_val) {
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t slice = gtid >> 5;
    if (slice >= nslices) return;
    const uint32_t p0 = gtid < nrows ? ptr[gtid] : 0u;
    const uint32_t len = gtid < nrows ? ptr[gtid + 1] - p0 : 0u;
    const uint64_t base = (uint64_t)slice_ptr[slice] * 32u + lane_id();
    const uint32_t width = slice_ptr[slice + 1] - slice_ptr[slice];
    for (uint32_t k = 0; k < width; ++k) {
        const bool real = k < len;
        slice_ind[base + (uint64_t)k * 32u] = real ? ind[p0 + k] : 0u;
        slice_val[base + (uint64_t)k * 32u] = real ? val[p0 + k] : (T)0;
    }
}

template <typename T, typename XG>
__global__ void __launch_bounds__(256, 8)
spmv_sliced_kernel(uint32_t nrows, uint32_t nslices, const uint32_t *__restrict__ ptr,
                   const uint32_t *__restrict__ slice_ptr, const uint32_t *__restrict__ slice_ind,
                   const T *__restrict__ slice_val, const XG xg, T *__restrict__ y) {
    constexpr int U = 4;   // entries in flight per lane
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t slice = row >> 5;
    if (slice >= nslices) return;
    const uint32_t len = row < nrows ? __ldg(ptr + row + 1) - __ldg(ptr + row) : 0u;
    const uint32_t s0 = __ldg(slice_ptr + slice), width = __ldg(slice_ptr + slice + 1) - s0;
    const uint32_t *__restrict__ ci = slice_ind + (uint64_t)s0 * 32u + lane_id();
    const T *__restrict__ cv = slice_val + (uint64_t)s0 * 32u + lane_id();
    T acc = (T)0;
    for (uint32_t k = 0; k < width; k += U) {
        uint32_t c[U];
        T v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t ku = k + u < width ? k + u : k;      // k itself is in range: safe dummy
            c[u] = __ldg(ci + (uint64_t)ku * 32u);
            v[u] = __ldg(cv + (uint64_t)ku * 32u);
        }
        T xv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) xv[u] = k + u < len ? xg(c[u]) : (T)0;
#pragma unroll
        for (int u = 0; u < U; ++u) acc += k + u < len ? v[u] * xv[u] : (T)0;     // ascending column order
    }
    if (row < nrows) y[row] = acc;
}

// Builds the sliced copy if the padding stays within `max_ratio` of the stored entries; returns
// whether it exists afterwards.  Caller holds a->plan_mu.
template <typename T>
bool build_slices(spl_ctx *ctx, spl_mat *a, double max_ratio) {
    if (a->slice_ptr) return true;
    if (a->nnz == 0) return false;
    const uint32_t nslices = div_up(a->nrows, 32);
    Tmp<uint32_t> width(ctx, nslices);
    Tmp<uint32_t> sp(ctx, (size_t)nslices + 1);
    slice_width_kernel<<<div_up((uint64_t)nslices * 32, 256), 256, 0, ctx->stream>>>(a->ptr, a->nrows, nslices, width);
    check_launch(ctx, "slice_width");
    exclusive_scan_u32(ctx, width, nslices, sp);
    uint32_t total_width = 0;
    read_back(ctx, sp.p + nslices, &total_width, 1);
    const uint64_t padded = (uint64_t)total_width * 32u;
    if ((double)padded > max_ratio * (double)a->nnz + 4096.0) return false;
    uint32_t *si = nullptr;
    T *sv = nullptr;
    if (cudaMallocFromPoolAsync((void **)&si, padded * sizeof(uint32_t), ctx->pool, ctx->stream) != cudaSuccess ||
        cudaMallocFromPoolAsync((void **)&sv, padded * sizeof(T), ctx->pool, ctx->stream) != cudaSuccess) {
        cudaGetLastError();                      // no room for a second copy: stay with CSR
        if (si) cudaFreeAsync(si, ctx->stream);
        return false;
    }
    slice_fill_kernel<T><<<div_up((uint64_t)nslices * 32, 256), 256, 0, ctx->stream>>>(
        a->ptr, a->ind, static_cast<const T *>(a->val), a->nrows, nslices, sp, si, sv);
    check_launch(ctx, "slice_fill");
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    a->slice_ind = si;
    a->slice_val = sv;
    a->slice_entries = padded;
    a->slice_ptr = sp.release();
    return true;
}

template <typename T, typename XG>
void spmv_sliced(spl_ctx *ctx, const spl_mat *a, const XG &xg, T *y) {
    const uint32_t nslices = div_up(a->nrows, 32);
    spmv_sliced_kernel<T, XG><<<div_up((uint64_t)nslices * 32, 256), 256, 0, ctx->stream>>>(
        a->nrows, nslices, a->ptr, a->slice_ptr, a->slice_ind, static_cast<const T *>(a->slice_val), xg, y);
    check_launch(ctx, "spmv_sliced");
}

// ------------------------------------------------------------------ merge-path kernel
// Merge path over A = row end offsets ptr[1..nrows] and B = 0..nnz-1 (Merrill & Garland): the
// path has nrows + nnz items; tile t owns items [t*ITEMS, (t+1)*ITEMS).  The tile start
// coordinates depend on the matrix only and are cached in the plan (spl_mat::merge_rows).
// Inside a tile: (1) the tile's nnz are streamed with 128-bit coalesced loads, multiplied by the
// gathered x and parked in shared memory; (2) every thread walks IPT consecutive path items
// from shared memory (balanced whatever the row lengths), writes the rows it finishes, and
// (3) a segmented warp-shuffle scan hands the partial sum of a row that spans threads to the
// thread that finishes it.  The row still open at the tile end goes to a per-tile carry that
// spmv_merge_fixup_kernel adds in tile order (deterministic, no atomics).
constexpr int MG_THREADS = 256;

__global__ void merge_partition_kernel(const uint32_t *__restrict__ ptr, uint32_t nrows, uint32_t nnz,
                                       uint32_t items, uint32_t ntiles,
                                       uint32_t *__restrict__ tile_rows) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > ntiles) return;
    const uint64_t total = (uint64_t)nrows + nnz;
    uint64_t d = (uint64_t)t * items;
    if (d > total) d = total;
    uint64_t lo = d > nnz ? d - nnz : 0, hi = d < nrows ? d : nrows;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if ((uint64_t)__ldg(ptr + mid + 1) <= d - mid - 1) lo = mid + 1;
        else hi = mid;
    }
    tile_rows[t] = (uint32_t)lo;
}

template <typename T, int IPT>
__global__ void __launch_bounds__(MG_THREADS)
spmv_merge_kernel(uint32_t nrows, uint32_t nnz, const uint32_t *__restrict__ ptr,
                  const uint32_t *__restrict__ ind, const T *__restrict__ val,
                  const T *__restrict__ x, T *__restrict__ y,
                  const uint32_t *__restrict__ tile_rows, uint32_t *__restrict__ carry_row,
                  T *__restrict__ carry_val) {
    constexpr int ITEMS = MG_THREADS * IPT;
    __shared__ __align__(16) T s_val[ITEMS + 8];           // values, then products, of the tile slice
    __shared__ __align__(16) uint32_t s_ind[ITEMS + 8];
    __shared__ uint32_t s_end[ITEMS + 1];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ T s_wval[MG_THREADS / 32];
    __shared__ int s_wflag[MG_THREADS / 32];

    const uint32_t tile = blockIdx.x;
    const uint64_t total = (uint64_t)nrows + nnz;
    const uint64_t d0 = (uint64_t)tile * ITEMS;
    const uint64_t d1 = d0 + ITEMS < total ? d0 + ITEMS : total;
    const uint32_t r0 = __ldg(tile_rows + tile), r1 = __ldg(tile_rows + tile + 1);
    const uint32_t z0 = (uint32_t)(d0 - r0), z1 = (uint32_t)(d1 - r1);
    const uint32_t t_rows = r1 - r0, t_nnz = z1 - z0, t_items = (uint32_t)(d1 - d0);

    // (1a) TMA: the 16-byte aligned superset [za, zb) of the tile's slice, one bulk copy per array
    const uint32_t za = z0 & ~3u, zb = (z1 + 3u) & ~3u;     // arrays carry 16 entries of slack
    const uint32_t shift = z0 - za;
    if (threadIdx.x == 0) {
        mbar_init(&s_bar, 1);
        mbar_init_fence();
    }
    __syncthreads();
    if (threadIdx.x == 0 && zb > za) {
        mbar_expect_tx(&s_bar, (zb - za) * (uint32_t)(sizeof(uint32_t) + sizeof(T)));
        tma_bulk_g2s(s_ind, ind + za, (zb - za) * (uint32_t)sizeof(uint32_t), &s_bar);
        tma_bulk_g2s(s_val, val + za, (zb - za) * (uint32_t)sizeof(T), &s_bar);
    }
    // (1b) row ends of the tile; the sentinel keeps the open row "unfinished"
    for (uint32_t i = threadIdx.x; i < t_rows; i += MG_THREADS) s_end[i] = __ldg(ptr + r0 + 1 + i);
    if (threadIdx.x == 0) s_end[t_rows] = 0xffffffffu;
    // (1c) products in place: consecutive lanes take consecutive entries, so neighbouring columns
    // share gather sectors; all IPT gathers of a thread are independent and in flight together
    if (zb > za) mbar_wait(&s_bar, 0);
    T *s_prod = s_val + shift;
    {
        T xv[IPT];
#pragma unroll
        for (int q = 0; q < IPT; ++q) {
            const uint32_t k = threadIdx.x + q * MG_THREADS;
            xv[q] = k < t_nnz ? __ldg(x + s_ind[shift + k]) : (T)0;
        }
#pragma unroll
        for (int q = 0; q < IPT; ++q) {
            const uint32_t k = threadIdx.x + q * MG_THREADS;
            if (k < t_nnz) s_prod[k] *= xv[q];
        }
    }
    __syncthreads();

    // (2) per-thread walk of IPT path items
    uint32_t dt = threadIdx.x * IPT;
    if (dt > t_items) dt = t_items;
    uint32_t lo = dt > t_nnz ? dt - t_nnz : 0, hi = dt < t_rows ? dt : t_rows;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (s_end[mid] <= z0 + (dt - mid - 1)) lo = mid + 1;
        else hi = mid;
    }
    uint32_t i = lo, j = dt - lo;
    T sum = (T)0, first_sum = (T)0;
    uint32_t first_row = 0;
    int hit = 0;
    uint32_t steps = t_items - dt < (uint32_t)IPT ? t_items - dt : (uint32_t)IPT;
    uint32_t row_end = s_end[i];
    for (uint32_t k = 0; k < steps; ++k) {
        if (z0 + j < row_end) {
            sum += s_prod[j];
            ++j;
        } else {
            if (!hit) { first_sum = sum; first_row = i; hit = 1; }
            else y[r0 + i] = sum;
            sum = (T)0;
            ++i;
            row_end = s_end[i];
        }
    }

    // (3) segmented scan of (hit, tail) across the block: c_t = partial of the row open at the
    // start of thread t, contributed by the preceding threads
    T v = sum;
    int f = hit;
    const unsigned lane = lane_id(), warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T pv = __shfl_up_sync(0xffffffffu, v, o);
        const int pf = __shfl_up_sync(0xffffffffu, f, o);
        if (lane >= (unsigned)o) {
            if (!f) v += pv;
            f |= pf;
        }
    }
    if (lane == 31) { s_wval[warp] = v; s_wflag[warp] = f; }
    T ev = __shfl_up_sync(0xffffffffu, v, 1);       // exclusive inside the warp
    int ef = __shfl_up_sync(0xffffffffu, f, 1);
    if (lane == 0) { ev = (T)0; ef = 0; }
    __syncthreads();
    T pv = (T)0;                                     // carry entering this warp
    for (unsigned w = 0; w < warp; ++w) pv = s_wflag[w] ? s_wval[w] : pv + s_wval[w];
    const T carry_in = ef ? ev : pv + ev;
    if (hit) y[r0 + first_row] = first_sum + carry_in;
    if (threadIdx.x == MG_THREADS - 1) {
        carry_row[tile] = r1;                        // row still open at the tile end (== nrows: none)
        carry_val[tile] = f ? v : pv + v;
    }
}

template <typename T>
__global__ void spmv_merge_fixup_kernel(uint32_t nrows, uint32_t ntiles,
                                        const uint32_t *__restrict__ carry_row,
                                        const T *__restrict__ carry_val, T *__restrict__ y) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntiles) return;
    const uint32_t row = carry_row[t];
    if (row >= nrows) return;
    if (t > 0 && carry_row[t - 1] == row) return;    // the first tile of a run does the whole run
    T acc = (T)0;
    for (uint32_t u = t; u < ntiles && carry_row[u] == row; ++u) acc += carry_val[u];
    y[row] += acc;
}

template <typename T>
constexpr int merge_ipt() { return sizeof(T) == 8 ? 7 : 11; }   // odd: path walks stay off one bank

template <typename T>
void spmv_merge(spl_ctx *ctx, const spl_mat *a, const T *x, T *y) {
    constexpr int IPT = merge_ipt<T>();
    const uint32_t ntiles = a->merge_tiles;
    if (ntiles == 0) return;
    Tmp<uint32_t> carry_row(ctx, ntiles);
    Tmp<T> carry_val(ctx, ntiles);
    spmv_merge_kernel<T, IPT><<<ntiles, MG_THREADS, 0, ctx->stream>>>(
        a->nrows, a->nnz, a->ptr, a->ind, static_cast<const T *>(a->val), x, y, a->merge_rows,
        carry_row, carry_val);
    check_launch(ctx, "spmv_merge");
    spmv_merge_fixup_kernel<T><<<div_up(ntiles, 256), 256, 0, ctx->stream>>>(a->nrows, ntiles, carry_row,
                                                                            carry_val, y);
    check_launch(ctx, "spmv_merge_fixup");
}

// ------------------------------------------------------------------ stream kernel
// Persistent CTAs, the matrix stream decoupled from the threads that use it.  The vector kernel
// hides DRAM latency with resident threads: every lane's chain ptr -> col/val -> x is three
// dependent round trips, and an 80 MB matrix (config 1) is over before the pipeline is full.  Here
// every CTA owns one contiguous range of rows (ranges balanced on rows + stored entries, so all CTAs
// finish together) and walks it in tiles of R = CONS / LPR rows.  A tile's col/val entries are one
// contiguous slice of the CSR arrays, so ONE producer thread per CTA fetches it with two TMA bulk
// copies (cp.async.bulk, completion on an mbarrier) into a ring of S shared-memory stages, ahead of
// the consumer warps: the bytes in flight cost no registers.  The consumers read indices and values
// from shared memory, gather x (LPR lanes per row, U gathers in flight per lane), reduce, and free
// the stage (empty barrier).
//   * x: the producer also prefetches the leading edge of x into L2 (cp.async.bulk.prefetch.L2):
//     for banded / stencil matrices the only x bytes a tile touches first are those above the
//     largest column of the tiles before it, which the plan recorded per tile; the consumers'
//     gathers then hit L2 (or L1: consecutive tiles of a CTA overlap) instead of waiting on HBM.
//   * programmatic dependent launch: behind another product of this kind the kernel is launched with
//     cudaLaunchAttributeProgrammaticStreamSerialization; producers start their matrix prefetch at
//     once (the matrix is immutable), consumers wait (griddepcontrol.wait) before the first x gather
//     and y store, then release the next launch (griddepcontrol.launch_dependents).  Back-to-back
//     products (solver iterations) overlap one product's ramp with the tail of the one before.
//   * lanes take the entries of a row exactly as the vector kernel does, so the two kernels give the
//     same bits; with one lane per row the row sum runs in ascending column order: bit-identical to
//     the reference's `&A * &X` (src/csr/ops/mul.rs:25-40).
// The tile layout and the consumers' row loop are those of stream_tile.cuh (shared with the fused
// gather kernel, gather.cu); the copy and barrier primitives are those of ptx.cuh.
constexpr uint32_t kStreamXEdgeMax = 1u << 15;     // longest leading edge of x one tile prefetches (elements)

// largest number of stored entries in any window of `rows` consecutive rows (bounds every tile)
__global__ void stream_window_kernel(const uint32_t *__restrict__ ptr, uint32_t nrows, uint32_t rows,
                                     uint32_t *__restrict__ max_window) {
    uint32_t m = 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e = r + rows < nrows ? r + rows : nrows;
        m = max(m, ptr[e] - ptr[r]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane_id() == 0 && m) atomicMax(max_window, m);
}

// cta_rows[b] = first row of CTA b: the smallest r with ptr[r] + r >= b * (nnz + nrows) / grid, rounded
// down to a multiple of 4 rows (the pointer slice of a tile is fetched by a 16-byte aligned bulk copy)
__global__ void stream_partition_kernel(const uint32_t *__restrict__ ptr, uint32_t nrows, uint32_t nnz, uint32_t grid,
                                        uint32_t rows_per_tile, uint32_t *__restrict__ cta_rows,
                                        uint32_t *__restrict__ max_tiles) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > grid) return;
    auto first_row = [&](uint32_t q) -> uint32_t {
        if (q == 0) return 0u;
        if (q >= grid) return nrows;
        const uint64_t target = ((uint64_t)nnz + nrows) * q / grid;
        uint32_t lo = 0, hi = nrows;
        while (lo < hi) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            if ((uint64_t)__ldg(ptr + mid) + mid < target) lo = mid + 1;
            else hi = mid;
        }
        return lo & ~3u;
    };
    const uint32_t r0 = first_row(b);
    cta_rows[b] = r0;
    if (b < grid) atomicMax(max_tiles, (first_row(b + 1) - r0 + rows_per_tile - 1) / rows_per_tile);
}

// The matrix's row pattern as a kernel parameter (spl_mat::pattern_off / pattern_len; len 0: none).
struct RowPattern {
    uint32_t off[kPatternMax];
    uint32_t len;
};

// Per CTA b, slots [b * (max_tiles + 1) ...]: tile_lo[k] = position of tile k's first stored entry
// (k = number of tiles: the end of the range); xhi[k] = 1 + the largest column of tile k (rows are
// column-sorted: the last entry of a row), 0 if the tile has no entry; xlo0[b] = the smallest column of
// the CTA's first tile.  With a row pattern: reg[k] = 1 when tile k is regular (every row r has pat.len
// entries at columns r + pat.off[j]), and *regular counts the regular tiles of the grid.  reg and xhi
// arrive zeroed.
__global__ void stream_edges_kernel(const uint32_t *__restrict__ ptr, const uint32_t *__restrict__ ind,
                                    const uint32_t *__restrict__ cta_rows, uint32_t rows_per_tile, uint32_t max_tiles,
                                    uint32_t *__restrict__ tile_lo, uint32_t *__restrict__ xhi,
                                    uint32_t *__restrict__ xlo0, const __grid_constant__ RowPattern pat,
                                    uint32_t *__restrict__ reg, uint32_t *__restrict__ regular) {
    const uint32_t b = blockIdx.x;
    const uint32_t rs = cta_rows[b], re = cta_rows[b + 1];
    const size_t base = (size_t)b * (max_tiles + 1);
    for (uint32_t k = threadIdx.x; k <= max_tiles; k += blockDim.x) {
        const uint64_t r = (uint64_t)rs + (uint64_t)k * rows_per_tile;
        tile_lo[base + k] = ptr[r < re ? r : re];
    }
    for (uint32_t r = rs + threadIdx.x; r < re; r += blockDim.x) {
        const uint32_t lo = ptr[r], hi = ptr[r + 1];
        const uint32_t k = (r - rs) / rows_per_tile;
        if (pat.len) {                                  // reg[] holds "irregular" until the pass below
            bool fits = hi - lo == pat.len;
            for (uint32_t j = 0; fits && j < pat.len; ++j) fits = ind[lo + j] == r + pat.off[j];
            if (!fits) reg[base + k] = 1u;
        }
        if (hi == lo) continue;
        atomicMax(xhi + base + k, ind[hi - 1] + 1u);
        if (k == 0) atomicMin(xlo0 + b, ind[lo]);
    }
    if (!pat.len) return;
    __syncthreads();
    const uint32_t ntiles = (re - rs + rows_per_tile - 1) / rows_per_tile;
    uint32_t count = 0;
    for (uint32_t k = threadIdx.x; k < ntiles; k += blockDim.x) {
        const uint32_t fits = reg[base + k] ^ 1u;
        reg[base + k] = fits;
        count += fits;
    }
    if (count) atomicAdd(regular, count);
}

// TIGHT: registers held to 56 so that four CTAs fit on an SM; otherwise three CTAs with room for
// eight f64 gathers and values in flight per lane.
// PAT: the grid has regular tiles (stream_edges_kernel).  Their columns and row starts follow from the row
// number and the row pattern, so the producer fetches only their values; the consumers take column
// r + pat.off[j] for position j of row r, and everything else runs as on any tile (same bits).
template <typename T, int LPR, int U, bool TIGHT, bool PAT, typename XG>
__global__ void __launch_bounds__(TILE_CONSUMERS + 32, TIGHT ? 4 : 3)
spmv_stream_kernel(uint32_t nrows, const uint32_t *__restrict__ ptr, const uint32_t *__restrict__ ind,
                   const T *__restrict__ val, const XG xg, T *__restrict__ y, const uint32_t *__restrict__ cta_rows,
                   const uint32_t *__restrict__ tile_lo, const uint32_t *__restrict__ xhi,
                   const uint32_t *__restrict__ xlo0, uint32_t max_tiles, uint32_t cap, uint32_t stages,
                   const T *__restrict__ x_edge, uint32_t x_lo, uint32_t x_hi, int l2_hint,
                   const uint32_t *__restrict__ tile_reg, const __grid_constant__ RowPattern pat) {
    constexpr uint32_t CONS = TILE_CONSUMERS;
    constexpr uint32_t R = tile_rows(LPR), PTRS = tile_ptr_slots(R);
    extern __shared__ __align__(128) unsigned char st_raw[];
    // per stage: [cap] indices, [cap] values, [PTRS] row pointers; then the barriers; with PAT one word per
    // stage (the first entry position of a regular tile, ~0 for any other) and the row pattern
    uint32_t *s_ind = reinterpret_cast<uint32_t *>(st_raw);
    T *s_val = reinterpret_cast<T *>(st_raw + (size_t)stages * cap * sizeof(uint32_t));
    uint32_t *s_ptr = reinterpret_cast<uint32_t *>(st_raw + (size_t)stages * cap * (sizeof(uint32_t) + sizeof(T)));
    uint64_t *full = reinterpret_cast<uint64_t *>(s_ptr + (size_t)stages * PTRS);
    uint64_t *empty = full + stages;
    uint32_t *s_reg_lo = reinterpret_cast<uint32_t *>(empty + stages);
    uint32_t *s_pat = s_reg_lo + stages;
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < stages; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, CONS / 32);
        }
        mbar_init_fence();
    }
    if (PAT && threadIdx.x < pat.len) s_pat[threadIdx.x] = pat.off[threadIdx.x];
    __syncthreads();
    const uint32_t rs = __ldg(cta_rows + blockIdx.x), re = __ldg(cta_rows + blockIdx.x + 1);
    const uint32_t ntiles = (re - rs + R - 1) / R;

    if (threadIdx.x >= CONS) {
        // ---- producer: one thread, up to S tiles ahead of the consumers ----
        if (threadIdx.x != CONS || ntiles == 0) return;
        const size_t base = (size_t)blockIdx.x * (max_tiles + 1);
        const uint32_t *t_lo = tile_lo + base, *t_xhi = xhi + base, *t_reg = tile_reg + base;
        uint32_t s = 0, phase = 0;
        uint32_t edge = __ldg(xlo0 + blockIdx.x);                 // x below this is somebody else's first touch
        uint32_t lo = __ldg(t_lo);
        const uint64_t pol = l2_policy_evict_first();
        for (uint32_t k = 0; k < ntiles; ++k) {
            const uint32_t hi = __ldg(t_lo + k + 1), x1 = __ldg(t_xhi + k);     // consecutive words: L1 hits
            if (k >= stages) mbar_wait(empty + s, phase ^ 1u);     // the consumers are done with this stage
            const uint32_t za = slice_lo(lo), cnt = slice_hi(hi) - za;
            // a regular tile: no pointer or index slice, its first entry position goes through the stage
            const bool regular = PAT && __ldg(t_reg + k);
            if (PAT) s_reg_lo[s] = regular ? lo : ~0u;             // published by the arrive below (release)
            const uint32_t r0 = rs + k * R;                        // multiple of 4
            const uint32_t left = (nrows + 1u - r0 + 3u) & ~3u;    // pointer entries from r0 to the end (+ slack)
            const uint32_t np = regular ? 0u : left < PTRS ? left : PTRS;
            const uint32_t ni = regular ? 0u : cnt;
            mbar_expect_tx(full + s, ni * (uint32_t)sizeof(uint32_t) + cnt * (uint32_t)sizeof(T) + np * (uint32_t)sizeof(uint32_t));
            if (np) tma_bulk_g2s(s_ptr + (size_t)s * PTRS, ptr + r0, np * (uint32_t)sizeof(uint32_t), full + s);
            if (cnt && l2_hint) {
                if (ni) tma_bulk_g2s_hint(s_ind + (size_t)s * cap, ind + za, ni * (uint32_t)sizeof(uint32_t), full + s, pol);
                tma_bulk_g2s_hint(s_val + (size_t)s * cap, val + za, cnt * (uint32_t)sizeof(T), full + s, pol);
            } else if (cnt) {
                if (ni) tma_bulk_g2s(s_ind + (size_t)s * cap, ind + za, ni * (uint32_t)sizeof(uint32_t), full + s);
                tma_bulk_g2s(s_val + (size_t)s * cap, val + za, cnt * (uint32_t)sizeof(T), full + s);
            }
            if (x_edge && x1 > edge) {                             // leading edge of x -> L2
                // the part of (edge, x1] that lives in the local array x_edge[x_lo, x_hi), in whole 16-byte units
                const uint32_t a = edge > x_lo ? edge : x_lo, b = x1 < x_hi ? x1 : x_hi;
                if (b > a && b - a <= kStreamXEdgeMax) {
                    const uintptr_t end = reinterpret_cast<uintptr_t>(x_edge + x_hi) & ~(uintptr_t)15;
                    const uintptr_t p0 = reinterpret_cast<uintptr_t>(x_edge + a) & ~(uintptr_t)15;
                    uintptr_t p1 = (reinterpret_cast<uintptr_t>(x_edge + b) + 15) & ~(uintptr_t)15;
                    if (p1 > end) p1 = end;
                    if (p1 > p0) l2_prefetch_bulk(reinterpret_cast<const void *>(p0), (uint32_t)(p1 - p0));
                }
                edge = x1;
            }
            lo = hi;
            if (++s == stages) { s = 0; phase ^= 1u; }
        }
        return;
    }

    // ---- consumers: CONS threads, LPR lanes per row; nothing but x comes from global memory ----
    const uint32_t rl = threadIdx.x / LPR, sub = threadIdx.x % LPR;
    uint32_t s = 0, phase = 0;
    griddep_wait();                    // x (and y's previous readers) belong to the launch before this one
    if (threadIdx.x == 0) griddep_launch();
    for (uint32_t k = 0; k < ntiles; ++k) {
        mbar_wait(full + s, phase);
        const uint32_t *cp = s_ptr + (size_t)s * PTRS;
        const uint32_t *ci = s_ind + (size_t)s * cap;
        const T *cv = s_val + (size_t)s * cap;
        const uint32_t r = rs + k * R + rl;
        // column of stage position j: cb[j] + cadd (a regular tile: cb = the pattern moved to the row's start)
        const uint32_t *cb = ci;
        uint32_t cadd = 0, p0 = 0, e = 0;
        const uint32_t reg_lo = PAT ? s_reg_lo[s] : ~0u;
        if (reg_lo != ~0u) {
            if (r < re) { p0 = (reg_lo & 3u) + rl * pat.len; e = p0 + pat.len; cb = s_pat - p0; cadd = r; }
        } else {
            const uint32_t za = slice_lo(cp[0]);
            if (r < re) { p0 = cp[rl] - za; e = cp[rl + 1] - za; }
        }
        T acc = (T)0;
        // the row's columns are sorted: first and last entry bound them
        if (e <= p0 || xg.all_local(cb[p0] + cadd, cb[e - 1] + cadd))
            tile_row_sum<T, LPR, U>(acc, cb, cadd, cv, p0, e, sub, [&](uint32_t c) { return xg.local(c); });
        else
            tile_row_sum<T, LPR, U>(acc, cb, cadd, cv, p0, e, sub, [&](uint32_t c) { return xg(c); });
        __syncwarp();
        if (lane_id() == 0) mbar_arrive(empty + s);
        acc = row_lanes_sum<LPR>(acc);
        if (sub == 0 && r < re) y[r] = xg.poisoned() ? (T)NAN : acc;
        if (++s == stages) { s = 0; phase ^= 1u; }
    }
}

inline int env_int(const char *name, int fallback) {
    const char *e = std::getenv(name);
    return e ? std::atoi(e) : fallback;
}

inline size_t stream_stage_bytes(const spl_mat *a) {
    return (size_t)a->stream_cap * (4 + a->vsize()) + (size_t)tile_ptr_slots(a->stream_rows) * 4;
}
RowPattern row_pattern(const spl_mat *a) {
    RowPattern p{};
    std::memcpy(p.off, a->pattern_off, sizeof(p.off));
    p.len = a->pattern_len;
    return p;
}

// Largest window of R rows -> stage capacity in entries (0: a tile does not fit in shared memory).
// Caller holds a->plan_mu or is the planner.
void stream_capacity(spl_ctx *ctx, spl_mat *a, uint32_t rows_per_tile) {
    if (a->stream_rows == rows_per_tile) return;
    a->stream_rows = rows_per_tile;
    a->stream_cap = 0;
    a->stream_grid = 0;
    if (a->nnz == 0) return;
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch + 1, 0, sizeof(uint32_t), ctx->stream));
    stream_window_kernel<<<std::min<unsigned>(div_up(a->nrows, 256), (unsigned)ctx->num_sms * 8u), 256, 0, ctx->stream>>>(
        a->ptr, a->nrows, rows_per_tile, ctx->d_scratch + 1);
    check_launch(ctx, "stream_window");
    uint32_t max_window = 0;
    read_back(ctx, ctx->d_scratch + 1, &max_window, 1);
    const uint32_t cap = stage_capacity(max_window);
    // three stages of it (with the pointer slices) must fit beside the barriers
    if (3 * ((size_t)cap * (4 + a->vsize()) + ((size_t)rows_per_tile + 4) * 4) + 64 <= 226 * 1024) a->stream_cap = cap;
}

// Row range per CTA and the x edges per tile for a grid of `grid` CTAs.  Cached; rebuilt when the grid changes.
void stream_partition(spl_ctx *ctx, spl_mat *a, uint32_t grid) {
    if (a->stream_grid == grid) return;
    std::lock_guard<std::mutex> lock(a->plan_mu);
    if (a->stream_grid == grid) return;
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));                  // nobody is reading the old arrays
    dfree(ctx, a->stream_cta_rows); dfree(ctx, a->stream_xhi); dfree(ctx, a->stream_xlo0); dfree(ctx, a->stream_tile_lo);
    dfree(ctx, a->stream_tile_reg);
    a->stream_cta_rows = a->stream_xhi = a->stream_xlo0 = a->stream_tile_lo = a->stream_tile_reg = nullptr;
    a->stream_cta_rows = dalloc<uint32_t>(ctx, (size_t)grid + 1);
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch + 1, 0, sizeof(uint32_t), ctx->stream));
    stream_partition_kernel<<<div_up((uint64_t)grid + 1, 128), 128, 0, ctx->stream>>>(
        a->ptr, a->nrows, a->nnz, grid, a->stream_rows, a->stream_cta_rows, ctx->d_scratch + 1);
    check_launch(ctx, "stream_partition");
    uint32_t max_tiles = 0;
    read_back(ctx, ctx->d_scratch + 1, &max_tiles, 1);
    max_tiles = std::max(max_tiles, 1u);
    a->stream_max_tiles = max_tiles;
    const size_t slots = (size_t)grid * (max_tiles + 1);
    a->stream_xhi = dalloc<uint32_t>(ctx, slots);
    a->stream_tile_lo = dalloc<uint32_t>(ctx, slots);
    a->stream_xlo0 = dalloc<uint32_t>(ctx, grid);
    a->stream_tile_reg = dalloc<uint32_t>(ctx, slots);
    SPL_CUDA(cudaMemsetAsync(a->stream_xhi, 0, sizeof(uint32_t) * slots, ctx->stream));
    SPL_CUDA(cudaMemsetAsync(a->stream_xlo0, 0xff, sizeof(uint32_t) * (size_t)grid, ctx->stream));
    SPL_CUDA(cudaMemsetAsync(a->stream_tile_reg, 0, sizeof(uint32_t) * slots, ctx->stream));
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch + 1, 0, sizeof(uint32_t), ctx->stream));
    stream_edges_kernel<<<grid, 256, 0, ctx->stream>>>(a->ptr, a->ind, a->stream_cta_rows, a->stream_rows, max_tiles,
                                                      a->stream_tile_lo, a->stream_xhi, a->stream_xlo0, row_pattern(a),
                                                      a->stream_tile_reg, ctx->d_scratch + 1);
    check_launch(ctx, "stream_edges");
    read_back(ctx, ctx->d_scratch + 1, &a->stream_regular, 1);    // synchronises: visible to any other stream from here on
    a->stream_grid = grid;
}

// Sets the kernel's dynamic shared memory to `smem` and returns how many of its CTAs fit on an SM (cached per
// instantiation).
template <typename K>
uint32_t stream_resident(K k, size_t smem, std::atomic<size_t> &smem_set, std::atomic<uint64_t> &occ_cache) {
    if (smem > smem_set.load(std::memory_order_relaxed)) {
        SPL_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set.store(smem, std::memory_order_relaxed);
    }
    uint64_t oc = occ_cache.load(std::memory_order_relaxed);     // (smem << 8) | resident CTAs
    if ((oc >> 8) != smem) {
        int resident = 0;
        SPL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, k, TILE_CONSUMERS + 32, smem));
        SPL_REQUIRE(resident >= 1, SPL_ERR_CUDA, "stream SpMV: no CTA fits on an SM");
        oc = ((uint64_t)smem << 8) | (uint64_t)resident;
        occ_cache.store(oc, std::memory_order_relaxed);
    }
    return (uint32_t)(oc & 0xff);
}

// x_edge: array indexable by column over [x_lo, x_hi) in local memory (the whole x, or this rank's own
// slice of a sharded x with the pointer moved back by the slice's first column), or NULL
template <typename T, int LPR, int U, bool TIGHT, typename XG>
void launch_stream(spl_ctx *ctx, const spl_mat *a, const XG &xg, T *y, const T *x_edge, uint32_t x_lo, uint32_t x_hi) {
    auto k_csr = spmv_stream_kernel<T, LPR, U, TIGHT, false, XG>;
    auto k_pat = spmv_stream_kernel<T, LPR, U, TIGHT, true, XG>;
    constexpr int CONS = TILE_CONSUMERS;
    // shape (measured, profiles/r2_spmv_notes.md): three stages, three CTAs of 64 registers per SM; a
    // deeper ring or a fourth, register-starved CTA does not pay
    const size_t stage_bytes = stream_stage_bytes(a);
    const uint32_t stages = (uint32_t)std::max(2, env_int("SPL_STREAM_STAGES", 3));
    const size_t smem_csr = stages * stage_bytes + 2 * stages * sizeof(uint64_t);
    const size_t smem_pat = smem_csr + (stages + kPatternMax) * sizeof(uint32_t);
    SPL_REQUIRE(smem_csr <= 227 * 1024, SPL_ERR_UNSUPPORTED, "stream SpMV: the stages do not fit in shared memory");
    static std::atomic<size_t> smem_set_csr{0}, smem_set_pat{0};
    static std::atomic<uint64_t> occ_csr{0}, occ_pat{0};
    // the grid is the CSR kernel's: a matrix without regular tiles runs exactly that kernel, and the
    // partition (with the regular tiles) does not depend on which of the two kernels runs
    const uint32_t resident = stream_resident(k_csr, smem_csr, smem_set_csr, occ_csr);
    uint32_t ctas = (uint32_t)env_int("SPL_STREAM_CTAS", 0);
    if (ctas == 0 || ctas > resident) ctas = resident;
    const uint32_t grid = (uint32_t)ctx->num_sms * ctas;
    stream_partition(ctx, const_cast<spl_mat *>(a), grid);
    // regular tiles: the pattern kernel, on the same grid (SPL_STREAM_PATTERN=0 turns it off for A/B measurements).
    // It may need fewer registers than the CSR kernel (C1: 56 against 63), so one more of its CTAs could fit on
    // an SM; programmatic dependent launch then places the next product's CTAs there early, which was measured
    // slower (C1, one L2-resident copy: 12.7 against 11.0 us per product, profiles/r3_spmv_notes.md).  Its shared
    // memory is padded so that exactly the grid's CTAs per SM fit, as with the CSR kernel.
    bool pat = a->stream_regular && env_int("SPL_STREAM_PATTERN", 1) != 0;
    size_t smem_pat_run = smem_pat;
    if (pat) {
        static const size_t sm_bytes = [] {
            int dev = 0, per_sm = 0, reserved = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
            cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, dev);
            return ((size_t)per_sm << 16) | (size_t)reserved;
        }();
        const size_t per_sm = sm_bytes >> 16, reserved = sm_bytes & 0xffff;
        const size_t one_more = per_sm / (ctas + 1) + 1;            // ctas + 1 CTAs of this size do not fit
        if (one_more > reserved) smem_pat_run = std::max(smem_pat, std::min<size_t>(one_more - reserved, 227 * 1024));
        pat = smem_pat_run <= 227 * 1024 && stream_resident(k_pat, smem_pat_run, smem_set_pat, occ_pat) >= ctas;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(CONS + 32);
    cfg.dynamicSmemBytes = pat ? smem_pat_run : smem_csr;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (ctx->pdl_prev && !std::getenv("SPL_NO_PDL")) ? 1 : 0;     // only behind another stream-kernel product
    SPL_CUDA(cudaLaunchKernelEx(&cfg, pat ? k_pat : k_csr, a->nrows, (const uint32_t *)a->ptr, (const uint32_t *)a->ind,
                                static_cast<const T *>(a->val), xg, y, (const uint32_t *)a->stream_cta_rows,
                                (const uint32_t *)a->stream_tile_lo, (const uint32_t *)a->stream_xhi,
                                (const uint32_t *)a->stream_xlo0, a->stream_max_tiles, a->stream_cap, stages,
                                x_edge, x_lo, x_hi, env_int("SPL_STREAM_L2HINT", 1),
                                (const uint32_t *)a->stream_tile_reg, row_pattern(a)));
    check_launch(ctx, "spmv_stream");
    ctx->pdl_chain = true;
}

template <typename T, int LPR, typename XG>
void spmv_stream_u(spl_ctx *ctx, const spl_mat *a, const XG &xg, T *y, const T *x_edge, uint32_t x_lo, uint32_t x_hi) {
    // entries per lane and trip: one trip for the short rows of stencils and bands
    const bool wide = (a->max_row_len + LPR - 1) / LPR > 4;
    const bool tight = env_int("SPL_STREAM_TIGHT", 0) != 0;      // four CTAs of 56 registers: measured, not better
    if (wide) {
        if (tight) launch_stream<T, LPR, 8, true>(ctx, a, xg, y, x_edge, x_lo, x_hi);
        else launch_stream<T, LPR, 8, false>(ctx, a, xg, y, x_edge, x_lo, x_hi);
    } else {
        if (tight) launch_stream<T, LPR, 4, true>(ctx, a, xg, y, x_edge, x_lo, x_hi);
        else launch_stream<T, LPR, 4, false>(ctx, a, xg, y, x_edge, x_lo, x_hi);
    }
}

template <typename T, typename XG>
void spmv_stream(spl_ctx *ctx, const spl_mat *a, const XG &xg, T *y, const T *x_edge, uint32_t x_lo, uint32_t x_hi) {
    switch (a->plan_lanes) {
        case 1: spmv_stream_u<T, 1>(ctx, a, xg, y, x_edge, x_lo, x_hi); break;
        case 2: spmv_stream_u<T, 2>(ctx, a, xg, y, x_edge, x_lo, x_hi); break;
        case 4: spmv_stream_u<T, 4>(ctx, a, xg, y, x_edge, x_lo, x_hi); break;
        case 8: spmv_stream_u<T, 8>(ctx, a, xg, y, x_edge, x_lo, x_hi); break;
        case 16: spmv_stream_u<T, 16>(ctx, a, xg, y, x_edge, x_lo, x_hi); break;
        default: spmv_stream_u<T, 32>(ctx, a, xg, y, x_edge, x_lo, x_hi); break;
    }
}

template <typename T>
XPeer<T> make_xpeer(spl_ctx *ctx, const PeerX &px) {
    XPeer<T> xg;
    xg.world = px.world;
    for (int g = 0; g < SPL_MAX_PEERS; ++g) xg.slice[g] = static_cast<const T *>(px.slice[g]);
    for (int g = 0; g <= SPL_MAX_PEERS; ++g) xg.start[g] = px.start[g];
    xg.mine = xg.slice[px.rank];
    xg.my_start = px.start[px.rank];
    xg.my_len = px.start[px.rank + 1] - px.start[px.rank];
    xg.barrier_failed = ctx->d_scratch + 32;
    return xg;
}

template <typename T>
void spmv_peer_t(spl_ctx *ctx, const spl_mat *a, const PeerX &px, T *y, int lanes) {
    const XPeer<T> xg = make_xpeer<T>(ctx, px);
    if (a->plan_kernel == SPL_SPMV_STREAM && !std::getenv("SPL_PEER_VECTOR"))   // leading-edge prefetch inside the own slice
        spmv_stream<T>(ctx, a, xg, y, xg.mine - xg.my_start, xg.my_start, xg.my_start + xg.my_len);
    else spmv_vector<T>(ctx, a, xg, y, lanes, 0, a->nrows);
}

// ------------------------------------------------------------------ nnz-split kernel
// Merge-path's balance at warp granularity, without a block barrier: every warp owns a fixed chunk
// of K = 32*IPL consecutive stored entries, whatever the rows look like (a 700 000-entry row of a
// power-law matrix is just 2 700 chunks).  Lane l holds entries l, l+32, ... of the chunk: IPL
// coalesced col/val loads and then IPL independent x gathers are in flight per lane.  Rows are
// found from a per-chunk start row computed once per matrix (split_rows): rows [R0, R1) end inside
// the chunk (or are empty) and are written here, row R1 is still open at the chunk end and goes to
// the carry arrays, which a fix-up adds in chunk order (no atomics: run-to-run identical).
//   chunk inside one row  -> shuffle reduction straight from registers (the heavy-row fast path)
//   otherwise             -> products parked in the warp's 1 KB of shared memory, one lane per
//                            row; rows longer than 32 entries are summed by the whole warp.
// Only 8 KB of shared memory per CTA, so L1 keeps caching the hot columns of x.
constexpr int SP_THREADS = 256;
constexpr int SP_WARPS = SP_THREADS / 32;
template <typename T>
constexpr int split_ipl() { return sizeof(T) == 8 ? 4 : 8; }
constexpr int SP_FIX_SEQ = 32;        // carries one thread adds itself before handing the run to a CTA

__global__ void split_partition_kernel(const uint32_t *__restrict__ ptr, uint32_t nrows, uint32_t nnz,
                                       uint32_t chunk, uint32_t nchunks,
                                       uint32_t *__restrict__ chunk_row) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nchunks) return;
    // the row r with ptr[r] <= pos < ptr[r+1]  (pos < nnz, so it exists and is not empty)
    const uint32_t pos = w * chunk;
    chunk_row[w] = w == 0 ? 0u : upper_bound_u32(ptr, 0u, nrows + 1u, pos) - 1u;
}

constexpr uint32_t kHotFlag = 0x80000000u;   // column index = slot in the hot-column cache
constexpr uint32_t kHotBytes = 128 * 1024;    // shared memory given to the hot x values per CTA

// The registers of one chunk on one lane: IPL (index, value) pairs and the chunk's row range.
template <typename T, int IPL>
struct ChunkRegs {
    uint32_t c[IPL];
    T v[IPL];
    uint32_t R0, R1;
};

// Issues the loads of chunk w (coalesced, streaming) without using them: the hot kernel calls this one
// chunk ahead, so the col/val stream of the next chunk is in flight while this one's gathers are.
template <typename T, int IPL>
__device__ __forceinline__ void
split_load(ChunkRegs<T, IPL> &q, uint32_t w, uint32_t nrows, uint32_t nnz, uint32_t nchunks,
           const uint32_t *__restrict__ ind, const T *__restrict__ val, const uint32_t *__restrict__ chunk_row) {
    constexpr uint32_t K = 32 * IPL;
    const unsigned lane = lane_id();
    const uint32_t base = w * K;
    const uint32_t count = nnz - base < K ? nnz - base : K;
    q.R0 = __ldg(chunk_row + w);
    q.R1 = w + 1 == nchunks ? nrows : __ldg(chunk_row + w + 1);
#pragma unroll
    for (int u = 0; u < IPL; ++u) {
        const uint32_t j = lane + 32 * u;
        const uint32_t p = base + (j < count ? j : 0u);     // entry `base` exists: safe dummy
        q.c[u] = ld_stream(ind + p);
        q.v[u] = ld_stream(val + p);
    }
}

// One warp, one chunk.  HOT: indices carrying kHotFlag name a slot of the CTA's shared-memory copy of
// the hottest x values instead of a column.
template <typename T, int IPL, bool HOT>
__device__ __forceinline__ void
split_chunk(const ChunkRegs<T, IPL> &q, uint32_t w, uint32_t nrows, uint32_t nnz, uint32_t nchunks,
            const uint32_t *__restrict__ ptr, const T *__restrict__ x,
            T *__restrict__ y, uint32_t *__restrict__ carry_row,
            T *__restrict__ carry_val, T *sp, const T *s_hot) {
    constexpr uint32_t K = 32 * IPL;
    const unsigned lane = lane_id();
    const uint32_t base = w * K;
    const uint32_t count = nnz - base < K ? nnz - base : K;
    const bool last = w + 1 == nchunks;
    const uint32_t R0 = q.R0, R1 = q.R1;

    T prod[IPL];
#pragma unroll
    for (int u = 0; u < IPL; ++u)
        prod[u] = (HOT && (q.c[u] & kHotFlag)) ? s_hot[q.c[u] & ~kHotFlag] : __ldg(x + q.c[u]);
#pragma unroll
    for (int u = 0; u < IPL; ++u) prod[u] = lane + 32 * u < count ? q.v[u] * prod[u] : (T)0;

    if (R0 == R1) {          // the whole chunk lies inside the open row
        T s = prod[0];
#pragma unroll
        for (int u = 1; u < IPL; ++u) s += prod[u];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            carry_row[w] = R1;
            carry_val[w] = s;
        }
        return;
    }

#pragma unroll
    for (int u = 0; u < IPL; ++u) sp[lane + 32 * u] = prod[u];
    __syncwarp();
    for (uint32_t rb = R0; rb < R1; rb += 32) {
        const uint32_t r = rb + lane;
        const bool valid = r < R1;
        uint32_t lo = 0, hi = 0;
        if (valid) {
            lo = __ldg(ptr + r);
            hi = __ldg(ptr + r + 1) - base;          // ends inside the chunk: hi <= count
            lo = lo > base ? lo - base : 0u;         // the first row may have started earlier
        }
        const bool wide = hi - lo > 32u;
        if (valid && !wide) {
            T s = (T)0;
            for (uint32_t j = lo; j < hi; ++j) s += sp[j];
            y[r] = s;
        }
        unsigned todo = __ballot_sync(0xffffffffu, valid && wide);
        while (todo) {                               // rows of more than 32 entries: the whole warp adds
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint32_t l2 = __shfl_sync(0xffffffffu, lo, src), h2 = __shfl_sync(0xffffffffu, hi, src);
            T s = (T)0;
            for (uint32_t j = l2 + lane; j < h2; j += 32) s += sp[j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if ((int)lane == src) y[r] = s;
        }
    }
    // the row still open at the chunk end (none for the last chunk: every row ends by nnz)
    T s = (T)0;
    if (!last) {
        const uint32_t p1 = __ldg(ptr + R1);
        for (uint32_t j = (p1 > base ? p1 - base : 0u) + lane; j < count; j += 32) s += sp[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    }
    if (lane == 0) {
        carry_row[w] = R1;                           // == nrows for the last chunk: no carry
        carry_val[w] = s;
    }
}

template <typename T, int IPL>
__global__ void __launch_bounds__(SP_THREADS)
spmv_split_kernel(uint32_t nrows, uint32_t nnz, uint32_t nchunks, const uint32_t *__restrict__ ptr,
                  const uint32_t *__restrict__ ind, const T *__restrict__ val,
                  const T *__restrict__ x, T *__restrict__ y, const uint32_t *__restrict__ chunk_row,
                  uint32_t *__restrict__ carry_row, T *__restrict__ carry_val) {
    __shared__ T s_prod[SP_WARPS][32 * IPL];
    const uint32_t w = blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
    if (w >= nchunks) return;
    ChunkRegs<T, IPL> q;
    split_load<T, IPL>(q, w, nrows, nnz, nchunks, ind, val, chunk_row);
    split_chunk<T, IPL, false>(q, w, nrows, nnz, nchunks, ptr, x, y, carry_row, carry_val,
                               s_prod[threadIdx.x >> 5], nullptr);
}

// Hot-column variant: one persistent CTA per SM keeps the x values of the `nhot` hottest columns in
// shared memory (loaded once per launch through the hot-column list) and its warps walk the chunks
// with a grid stride, the col/val stream of the next chunk loaded (registers) while the gathers of
// the current one are in flight.  Gathers of hot columns never leave the SM.
template <typename T, int IPL, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
spmv_split_hot_kernel(uint32_t nrows, uint32_t nnz, uint32_t nchunks, const uint32_t *__restrict__ ptr,
                      const uint32_t *__restrict__ ind_hot, const T *__restrict__ val,
                      const T *__restrict__ x, T *__restrict__ y, const uint32_t *__restrict__ chunk_row,
                      uint32_t *__restrict__ carry_row, T *__restrict__ carry_val,
                      const uint32_t *__restrict__ hot_cols, uint32_t nhot) {
    extern __shared__ __align__(16) unsigned char sph_raw[];
    T *s_hot = reinterpret_cast<T *>(sph_raw);
    T *s_prod = s_hot + nhot;
    const uint32_t warp = threadIdx.x >> 5, warps = THREADS / 32;
    uint32_t w = blockIdx.x * warps + warp;
    const uint32_t stride = gridDim.x * warps;
    ChunkRegs<T, IPL> cur, nxt;
    if (w < nchunks) split_load<T, IPL>(cur, w, nrows, nnz, nchunks, ind_hot, val, chunk_row);   // under the table fill
    for (uint32_t j = threadIdx.x; j < nhot; j += THREADS) s_hot[j] = __ldg(x + __ldg(hot_cols + j));
    __syncthreads();
    while (w < nchunks) {
        const uint32_t wn = w + stride;
        if (wn < nchunks) split_load<T, IPL>(nxt, wn, nrows, nnz, nchunks, ind_hot, val, chunk_row);
        split_chunk<T, IPL, true>(cur, w, nrows, nnz, nchunks, ptr, x, y, carry_row, carry_val,
                                  s_prod + warp * (32 * IPL), s_hot);
        __syncwarp();          // the product buffer is reused by the warp's next chunk
        cur = nxt;
        w = wn;
    }
}

// Carries of one row sit in consecutive chunks.  The first chunk of a run adds the run in chunk
// order; runs longer than SP_FIX_SEQ are queued for a CTA each (fixed summation tree: deterministic).
template <typename T>
__global__ void spmv_split_fixup_kernel(uint32_t nrows, uint32_t nchunks,
                                        const uint32_t *__restrict__ carry_row,
                                        const T *__restrict__ carry_val, T *__restrict__ y,
                                        uint32_t *__restrict__ long_runs, uint32_t *__restrict__ n_long,
                                        uint32_t long_cap) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nchunks) return;
    const uint32_t row = carry_row[t];
    if (row >= nrows) return;
    if (t > 0 && carry_row[t - 1] == row) return;
    T acc = (T)0;
    uint32_t u = t;
    for (; u < nchunks && u < t + SP_FIX_SEQ && carry_row[u] == row; ++u) acc += carry_val[u];
    if (u < nchunks && u == t + SP_FIX_SEQ && carry_row[u] == row) {
        const uint32_t slot = atomicAdd(n_long, 1u);
        if (slot < long_cap) { long_runs[slot] = t; return; }
        for (; u < nchunks && carry_row[u] == row; ++u) acc += carry_val[u];     // queue full: finish here
    }
    y[row] += acc;
}

template <typename T>
__global__ void __launch_bounds__(256)
spmv_split_fixup_long_kernel(uint32_t nchunks, const uint32_t *__restrict__ carry_row,
                             const T *__restrict__ carry_val, T *__restrict__ y,
                             const uint32_t *__restrict__ long_runs, const uint32_t *__restrict__ n_long,
                             uint32_t long_cap) {
    __shared__ T s_part[8];
    __shared__ int s_more;
    const uint32_t n = min(*n_long, long_cap);
    for (uint32_t q = blockIdx.x; q < n; q += gridDim.x) {
        const uint32_t t = long_runs[q];
        const uint32_t row = carry_row[t];
        T acc = (T)0;
        for (uint32_t b = t;; b += 256) {            // 256 carries per trip until the run ends
            const uint32_t u = b + threadIdx.x;
            const bool in = u < nchunks && carry_row[u] == row;
            if (in) acc += carry_val[u];
            if (threadIdx.x == 0) s_more = 0;
            __syncthreads();
            if (threadIdx.x == 255 && in) s_more = 1;          // the run reaches past this trip
            __syncthreads();
            const int more = s_more;
            __syncthreads();
            if (!more) break;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane_id() == 0) s_part[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            T s = s_part[0];
            for (int k = 1; k < 8; ++k) s += s_part[k];
            y[row] += s;
        }
        __syncthreads();
    }
}

template <typename T>
void spmv_split(spl_ctx *ctx, const spl_mat *a, const T *x, T *y) {
    constexpr int IPL = split_ipl<T>();
    const uint32_t nchunks = a->split_chunks;
    if (nchunks == 0) {                              // no stored entry: y = 0
        SPL_CUDA(cudaMemsetAsync(y, 0, sizeof(T) * (size_t)a->nrows, ctx->stream));
        return;
    }
    constexpr uint32_t kLongCap = 1u << 16;
    Tmp<uint32_t> carry_row(ctx, nchunks);
    Tmp<T> carry_val(ctx, nchunks);
    Tmp<uint32_t> long_runs(ctx, kLongCap + 1);
    uint32_t *n_long = long_runs.p + kLongCap;
    SPL_CUDA(cudaMemsetAsync(n_long, 0, sizeof(uint32_t), ctx->stream));
    if (a->hot_state.load(std::memory_order_acquire) == 2 && a->ind_rank) {   // hot columns: persistent CTAs, hottest x values in shared memory
        const uint32_t nhot = a->hot_count;
        const char *te = std::getenv("SPL_HOT_THREADS");
        const int threads = te ? std::atoi(te) : 1024;
        const size_t smem = (size_t)nhot * sizeof(T) + (size_t)(threads / 32) * 32 * IPL * sizeof(T);
        auto go = [&](auto k) {
            SPL_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k<<<ctx->num_sms, threads, smem, ctx->stream>>>(
                a->nrows, a->nnz, nchunks, a->ptr, a->ind_rank, static_cast<const T *>(a->val), x, y,
                a->split_rows, carry_row, carry_val, a->col_order, nhot);
        };
        if (threads == 512) go(spmv_split_hot_kernel<T, IPL, 512>);
        else if (threads == 768) go(spmv_split_hot_kernel<T, IPL, 768>);
        else go(spmv_split_hot_kernel<T, IPL, 1024>);
        check_launch(ctx, "spmv_split_hot");
    } else {
        spmv_split_kernel<T, IPL><<<div_up(nchunks, SP_WARPS), SP_THREADS, 0, ctx->stream>>>(
            a->nrows, a->nnz, nchunks, a->ptr, a->ind, static_cast<const T *>(a->val), x, y, a->split_rows,
            carry_row, carry_val);
        check_launch(ctx, "spmv_split");
    }
    spmv_split_fixup_kernel<T><<<div_up(nchunks, 256), 256, 0, ctx->stream>>>(
        a->nrows, nchunks, carry_row, carry_val, y, long_runs, n_long, kLongCap);
    check_launch(ctx, "spmv_split_fixup");
    if (a->max_row_len > (uint32_t)(SP_FIX_SEQ * 32 * IPL)) {     // only then can a run exceed SP_FIX_SEQ
        spmv_split_fixup_long_kernel<T><<<ctx->num_sms * 2, 256, 0, ctx->stream>>>(
            nchunks, carry_row, carry_val, y, long_runs, n_long, kLongCap);
        check_launch(ctx, "spmv_split_fixup_long");
    }
}

// ------------------------------------------------------------------ hot-column renumbering
// A power-law matrix sends a large share of its gathers to a few thousand columns, but those sit
// one per 128-byte line of x, and L1 has tags for ~1 500 lines: ncu showed a 5 % L1 hit rate on the
// R-MAT matrix.  Renumbering the columns by how often they occur packs the hot part of x into a
// few hundred contiguous lines that L1 can hold.  Once per matrix: column histogram, stable sort by
// descending count, rank of every column, and a copy of the column indices in the new numbering.
// Per product: x is gathered into the new order (one pass over x), and the nnz-split kernel runs
// on (ind_rank, permuted x).  Rows are untouched, so y needs no fix-up.

__global__ void col_hist_kernel(const uint32_t *__restrict__ ind, uint32_t nnz, uint32_t *__restrict__ counts) {
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz;
         p += (uint64_t)gridDim.x * blockDim.x)
        atomicAdd(counts + ind[p], 1u);
}
// sort key: descending count = ascending (nrows - count); a column occurs at most once per row
struct LoadCountKey {
    const uint32_t *counts;
    uint32_t nrows;
    __device__ __forceinline__ uint32_t operator()(uint32_t i, uint32_t &) const { return nrows - counts[i]; }
};
struct LoadIota {
    __device__ __forceinline__ uint32_t operator()(uint32_t i, uint32_t &) const { return i; }
};
__global__ void hot_sum_kernel(const uint32_t *__restrict__ sorted_keys, uint32_t n, uint32_t nrows,
                               unsigned long long *__restrict__ out) {
    unsigned long long s = 0;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x)
        s += nrows - sorted_keys[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane_id() == 0 && s) atomicAdd(out, s);
}
// code[order[j]] = flag | j for the nhot hottest columns (j < nhot), the column itself otherwise
__global__ void hot_code_kernel(const uint32_t *__restrict__ order, uint32_t n, uint32_t nhot,
                                uint32_t *__restrict__ code) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) {
        const uint32_t c = order[j];
        code[c] = j < nhot ? (kHotFlag | j) : c;
    }
}
__global__ void renumber_kernel(const uint32_t *__restrict__ ind, uint32_t nnz, const uint32_t *__restrict__ rank,
                                uint32_t *__restrict__ out) {
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz;
         p += (uint64_t)gridDim.x * blockDim.x)
        out[p] = __ldg(rank + ind[p]);
}
void plan_hot_columns(spl_ctx *ctx, spl_mat *a) {
    const uint32_t ncols = a->ncols, nnz = a->nnz;
    const char *hot_kb = std::getenv("SPL_HOT_KB");        // table size (measurement knob); default 128 KB
    const uint32_t hot_bytes = hot_kb ? (uint32_t)std::atoi(hot_kb) * 1024u : kHotBytes;
    const uint32_t kHotColumns = hot_bytes / (uint32_t)a->vsize();      // 32 768 (f32) / 16 384 (f64) by default
    if (ncols < 4 * kHotColumns || nnz == 0) return;       // small x: nothing to gain
    Tmp<uint32_t> counts(ctx, ncols);
    SPL_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * (size_t)ncols, ctx->stream));
    const unsigned sgrid = (unsigned)ctx->num_sms * 16u;
    col_hist_kernel<<<sgrid, 256, 0, ctx->stream>>>(a->ind, nnz, counts);
    check_launch(ctx, "col_hist");
    Tmp<uint32_t> k0(ctx, ncols), k1(ctx, ncols), o0(ctx, ncols), o1(ctx, ncols);
    uint32_t *kb[2] = {k0, k1};
    uint32_t *ob[2] = {o0, o1};
    NoPayload *nb[2] = {nullptr, nullptr};
    const int r = radix_sort<uint32_t, uint32_t, NoPayload>(ctx, ncols, bits_for((uint64_t)a->nrows + 1),
                                                            LoadCountKey{counts, a->nrows}, LoadIota{},
                                                            LoadNone{}, kb, ob, nb);
    unsigned long long *sum = reinterpret_cast<unsigned long long *>(ctx->d_scratch + 2);
    SPL_CUDA(cudaMemsetAsync(sum, 0, sizeof(unsigned long long), ctx->stream));
    hot_sum_kernel<<<32, 256, 0, ctx->stream>>>(kb[r], kHotColumns, a->nrows, sum);
    check_launch(ctx, "hot_sum");
    uint32_t w[2];
    read_back(ctx, ctx->d_scratch + 2, w, 2);
    const double hot = (double)(((uint64_t)w[1] << 32) | w[0]);
    a->hot_coverage = hot / (double)nnz;
    if (std::getenv("SPL_DEBUG"))
        std::fprintf(stderr, "[spl] hot-column coverage of the %u hottest columns: %.3f\n", kHotColumns,
                     a->hot_coverage);
    if (a->hot_coverage < 0.2 || ncols >= kHotFlag) return;  // uniform columns: keep the plain indices
    a->hot_count = kHotColumns;
    a->col_order = dalloc<uint32_t>(ctx, kHotColumns);      // the hot columns, hottest first
    SPL_CUDA(cudaMemcpyAsync(a->col_order, ob[r], sizeof(uint32_t) * (size_t)kHotColumns,
                             cudaMemcpyDeviceToDevice, ctx->stream));
    uint32_t *code = ob[r ^ 1];                             // scratch: code[c] = c, or flag | slot if hot
    hot_code_kernel<<<div_up(ncols, 256), 256, 0, ctx->stream>>>(ob[r], ncols, kHotColumns, code);
    check_launch(ctx, "hot_code");
    a->ind_rank = dalloc<uint32_t>(ctx, (size_t)nnz + 16);
    renumber_kernel<<<sgrid, 256, 0, ctx->stream>>>(a->ind, nnz, code, a->ind_rank);
    check_launch(ctx, "renumber");
}

// ------------------------------------------------------------------ row statistics (plan)
// out[0] = longest row, out[1] = largest column, out[2] = ~smallest column (rows are column-sorted: the
// first and last entry of every row bound its columns)
__global__ void max_row_len_kernel(const uint32_t *__restrict__ ptr, const uint32_t *__restrict__ ind, uint32_t nrows,
                                   uint32_t *out) {
    uint32_t m = 0, cmax = 0, cmin_inv = 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrows;
         r += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t lo = ptr[r], hi = ptr[r + 1];
        m = max(m, hi - lo);
        if (hi > lo) {
            cmax = max(cmax, ind[hi - 1]);
            cmin_inv = max(cmin_inv, ~ind[lo]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
        cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
        cmin_inv = max(cmin_inv, __shfl_xor_sync(0xffffffffu, cmin_inv, o));
    }
    if (lane_id() == 0 && m) {
        atomicMax(out, m);
        atomicMax(out + 1, cmax);
        atomicMax(out + 2, cmin_inv);
    }
}

// *row = the first row in [from, nrows) with `len` entries (stays ~0 if there is none)
__global__ void pattern_row_kernel(const uint32_t *__restrict__ ptr, uint32_t from, uint32_t nrows, uint32_t len,
                                   uint32_t *row) {
    for (uint64_t r = from + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrows;
         r += (uint64_t)gridDim.x * blockDim.x) {
        if (ptr[r + 1] - ptr[r] == len) {        // a thread's first hit is its smallest: the minimum over threads is the first
            atomicMin(row, (uint32_t)r);
            return;
        }
    }
}

// The row pattern (spl_mat::pattern_off): the column offsets of the first row at or after nrows / 2 with the
// longest length, taken from the middle because the first rows of bands and stencils are boundary rows.
void plan_pattern(spl_ctx *ctx, spl_mat *a) {
    a->pattern_len = 0;
    const uint32_t len = a->max_row_len;
    if (len == 0 || len > kPatternMax) return;
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0xff, sizeof(uint32_t), ctx->stream));
    const uint32_t from = a->nrows / 2;
    pattern_row_kernel<<<std::min<unsigned>(div_up(a->nrows - from, 256), (unsigned)ctx->num_sms * 8u), 256, 0, ctx->stream>>>(
        a->ptr, from, a->nrows, len, ctx->d_scratch);
    check_launch(ctx, "pattern_row");
    uint32_t row = 0, p = 0;
    read_back(ctx, ctx->d_scratch, &row, 1);
    if (row == ~0u) return;
    read_back(ctx, a->ptr + row, &p, 1);
    read_back(ctx, a->ind + p, a->pattern_off, (int)len);
    for (uint32_t j = 0; j < len; ++j) a->pattern_off[j] -= row;
    a->pattern_len = len;
}

}  // namespace

void spmv_plan(spl_ctx *ctx, spl_mat *a) {
    if (a->plan_ready.load(std::memory_order_acquire)) return;
    std::lock_guard<std::mutex> lock(a->plan_mu);
    if (a->plan_ready.load(std::memory_order_relaxed)) return;
    uint32_t mx = 0;
    if (a->nnz) {
        SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, 3 * sizeof(uint32_t), ctx->stream));
        unsigned grid = min(div_up(a->nrows, 256), (unsigned)ctx->num_sms * 8u);
        max_row_len_kernel<<<grid, 256, 0, ctx->stream>>>(a->ptr, a->ind, a->nrows, ctx->d_scratch);
        check_launch(ctx, "max_row_len");
        uint32_t w[3] = {0, 0, 0};
        read_back(ctx, ctx->d_scratch, w, 3);
        mx = w[0];
        a->col_max = w[1];
        a->col_min = ~w[2];
    }
    a->max_row_len = mx;
    const double mean = a->nrows ? (double)a->nnz / a->nrows : 0.0;
    // lanes per row, from the measured sweeps (profiles/r1_spmv_notes.md): one lane up to ~12
    // entries per row (5- and 9-entry rows: 0.46 / 0.88-0.93 of peak against 0.42 / 0.75-0.85 with
    // two lanes), four lanes for 16..40 (random 16/row and the 27-point stencil), then one or two
    // trips of 4 in-flight entries per lane
    int lanes = 1;
    if (mean > 12.0) lanes = 4;
    while (lanes < 32 && lanes * 10 < mean) lanes *= 2;
    a->plan_lanes = lanes;
    // stream kernel: the largest window of 256 / lanes rows sizes its shared-memory stages; tiles that follow
    // the row pattern stream their values only
    stream_capacity(ctx, a, tile_rows(lanes));
    plan_pattern(ctx, a);
    // merge-path tile starts (matrix-only data, cached)
    const int ipt = a->dtype == SPL_F64 ? merge_ipt<double>() : merge_ipt<float>();
    const uint32_t items = MG_THREADS * ipt;
    const uint64_t total = (uint64_t)a->nrows + a->nnz;
    const uint32_t ntiles = div_up(total, items);
    a->merge_rows = dalloc<uint32_t>(ctx, (size_t)ntiles + 1);
    a->merge_tiles = ntiles;
    merge_partition_kernel<<<div_up((uint64_t)ntiles + 1, 256), 256, 0, ctx->stream>>>(
        a->ptr, a->nrows, a->nnz, items, ntiles, a->merge_rows);
    check_launch(ctx, "merge_partition");
    // nnz-split chunk start rows (matrix-only data, cached)
    const uint32_t chunk = 32u * (a->dtype == SPL_F64 ? split_ipl<double>() : split_ipl<float>());
    a->split_chunks = div_up(a->nnz, chunk);
    a->split_rows = dalloc<uint32_t>(ctx, (size_t)a->split_chunks + 1);
    if (a->split_chunks) {
        split_partition_kernel<<<div_up(a->split_chunks, 256), 256, 0, ctx->stream>>>(
            a->ptr, a->nrows, a->nnz, chunk, a->split_chunks, a->split_rows);
        check_launch(ctx, "split_partition");
    }
    // skewed rows (power law) -> balanced nnz-split kernel; regular rows -> vector
    const bool skewed = mean > 0 && (double)mx > 8.0 * mean + 64.0;
    a->plan_kernel = skewed ? SPL_SPMV_SPLIT : SPL_SPMV_VECTOR;
    // regular rows, a tile fits in shared memory and there is at least a tile per resident CTA: the
    // persistent stream kernel (same bits as the vector kernel: same lanes, same order)
    if (!skewed && a->stream_cap && (uint64_t)a->nrows * lanes >= (uint64_t)ctx->num_sms * 3u * TILE_CONSUMERS)
        a->plan_kernel = SPL_SPMV_STREAM;
    // the plan arrays were written on this context's stream: make them visible to any other stream
    SPL_CUDA(cudaStreamSynchronize(ctx->stream));
    a->plan_ready.store(1, std::memory_order_release);
}

// ------------------------------------------------------------------ CSC operands
// `&A * &X` with A a CscMatrix (src/csc/ops/mul.rs:5-61) accumulates every y[i] over ascending k, the
// same order as the row-wise product.  The CSC arrays are the CSR arrays of the transpose, so the
// row kernels cannot run on them; the first product on a CSC matrix builds its CSR form (one
// histogram + scan + scatter, recompress.cu) and keeps it with the matrix.  SPL_SPMV_SCATTER is the
// copy-free alternative: a lane group per column scatters val * x[col] into y with atomic adds
// (order of the adds not fixed: results vary in the last bits from run to run; tolerance parity only).
const spl_mat *csr_form(spl_ctx *ctx, const spl_mat *a) {
    if (a->format == SPL_CSR) return a;
    spl_mat *m = const_cast<spl_mat *>(a);
    if (spl_mat *t = m->twin.load(std::memory_order_acquire)) return t;
    std::lock_guard<std::mutex> lock(m->plan_mu);
    if (spl_mat *t = m->twin.load(std::memory_order_relaxed)) return t;
    spl_mat *t = new_mat(ctx, SPL_CSR, a->dtype, a->nrows, a->ncols, a->nnz);
    try {
        recompress(ctx, a->dtype, a->nmajor(), a->nminor(), a->nnz, a->ptr, a->ind, a->val, t->ptr, t->ind, t->val);
        publish_mat(ctx, t);
        SPL_CUDA(cudaStreamSynchronize(ctx->stream));          // visible to any other stream from here on
    } catch (...) {
        free_mat(ctx, t);
        throw;
    }
    m->twin.store(t, std::memory_order_release);
    return t;
}

void drop_value_copies(spl_ctx *ctx, spl_mat *m) {
    std::lock_guard<std::mutex> lock(m->plan_mu);
    free_mat(ctx, m->twin.exchange(nullptr));
    dfree(ctx, m->slice_ptr); dfree(ctx, m->slice_ind); dfree(ctx, m->slice_val);
    m->slice_ptr = m->slice_ind = nullptr;
    m->slice_val = nullptr;
    m->slice_entries = 0;
    m->slice_state.store(0, std::memory_order_release);
}

namespace {
template <typename T, int LPC>
__global__ void __launch_bounds__(256)
spmv_csc_scatter_kernel(uint32_t ncols, const uint32_t *__restrict__ ptr, const uint32_t *__restrict__ ind,
                        const T *__restrict__ val, const T *__restrict__ x, T *__restrict__ y) {
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t col = gtid / LPC;
    if (col >= ncols) return;
    const T xc = __ldg(x + col);
    const uint32_t e = __ldg(ptr + col + 1);
    for (uint32_t p = __ldg(ptr + col) + (uint32_t)(gtid % LPC); p < e; p += LPC)
        atomicAdd(y + __ldg(ind + p), __ldg(val + p) * xc);
}

template <typename T>
void spmv_csc_scatter(spl_ctx *ctx, const spl_mat *a, const T *x, T *y) {
    SPL_CUDA(cudaMemsetAsync(y, 0, sizeof(T) * (size_t)a->nrows, ctx->stream));
    if (a->nnz == 0) return;
    const double mean = (double)a->nnz / a->ncols;
    const T *v = static_cast<const T *>(a->val);
    if (mean <= 6.0)
        spmv_csc_scatter_kernel<T, 1><<<div_up(a->ncols, 256), 256, 0, ctx->stream>>>(a->ncols, a->ptr, a->ind, v, x, y);
    else if (mean <= 48.0)
        spmv_csc_scatter_kernel<T, 4><<<div_up((uint64_t)a->ncols * 4, 256), 256, 0, ctx->stream>>>(a->ncols, a->ptr, a->ind, v, x, y);
    else
        spmv_csc_scatter_kernel<T, 32><<<div_up((uint64_t)a->ncols * 32, 256), 256, 0, ctx->stream>>>(a->ncols, a->ptr, a->ind, v, x, y);
    check_launch(ctx, "spmv_csc_scatter");
}
}  // namespace

// x_lo / x_hi: the columns [x_lo, x_hi) of x that `x` (indexed by column) really holds; the whole vector
// unless the caller passed a window (spmv_window)
void spmv(spl_ctx *ctx, const spl_mat *a, const void *x, void *y, int kernel, int lanes, uint32_t x_lo, uint32_t x_hi) {
    if (x_hi == 0) x_hi = a->ncols;
    if (kernel == SPL_SPMV_SCATTER) {
        SPL_REQUIRE(a->format == SPL_CSC, SPL_ERR_UNSUPPORTED, "SPL_SPMV_SCATTER is the column kernel: it needs a CSC matrix");
        if (a->dtype == SPL_F32) spmv_csc_scatter<float>(ctx, a, (const float *)x, (float *)y);
        else spmv_csc_scatter<double>(ctx, a, (const double *)x, (double *)y);
        return;
    }
    a = csr_form(ctx, a);
    if (kernel == SPL_SPMV_AUTO) {
        spmv_plan(ctx, const_cast<spl_mat *>(a));
        kernel = a->plan_kernel;
        lanes = 0;
        // SPL_SPMV_KERNEL=vector|stream|split|merge overrides the planner (measurement / triage)
        const char *force = std::getenv("SPL_SPMV_KERNEL");
        if (force) {
            if (!std::strcmp(force, "vector")) kernel = SPL_SPMV_VECTOR;
            else if (!std::strcmp(force, "stream") && a->stream_cap) kernel = SPL_SPMV_STREAM;
            else if (!std::strcmp(force, "split")) kernel = SPL_SPMV_SPLIT;
            else if (!std::strcmp(force, "merge")) kernel = SPL_SPMV_MERGE;
        }
    }
    if (kernel == SPL_SPMV_STREAM) {
        spl_mat *m = const_cast<spl_mat *>(a);
        spmv_plan(ctx, m);
        if (a->stream_rows != tile_rows(a->plan_lanes)) {     // measurement knob changed
            std::lock_guard<std::mutex> lock(m->plan_mu);
            SPL_CUDA(cudaStreamSynchronize(ctx->stream));
            stream_capacity(ctx, m, tile_rows(a->plan_lanes));
        }
        SPL_REQUIRE(a->nnz == 0 || a->stream_cap, SPL_ERR_UNSUPPORTED,
                    "stream SpMV: a tile of rows does not fit in shared memory (skewed rows: use SPLIT)");
        if (a->nnz == 0) {
            SPL_CUDA(cudaMemsetAsync(y, 0, a->vsize() * (size_t)a->nrows, ctx->stream));
            return;
        }
        if (a->dtype == SPL_F32) spmv_stream<float>(ctx, a, XLocal<float>{(const float *)x}, (float *)y, (const float *)x, x_lo, x_hi);
        else spmv_stream<double>(ctx, a, XLocal<double>{(const double *)x}, (double *)y, (const double *)x, x_lo, x_hi);
        return;
    }
    if (kernel == SPL_SPMV_VECTOR && lanes == 0) {
        spmv_plan(ctx, const_cast<spl_mat *>(a));
        lanes = a->plan_lanes;
    }
    if (kernel == SPL_SPMV_SLICED) {     // forced: build the copy now, whatever the padding (within reason)
        spl_mat *m = const_cast<spl_mat *>(a);
        spmv_plan(ctx, m);
        if (m->slice_state.load(std::memory_order_acquire) != 2 || !m->slice_ptr) {
            std::lock_guard<std::mutex> lock(m->plan_mu);
            const bool ok = a->dtype == SPL_F32 ? build_slices<float>(ctx, m, 4.0) : build_slices<double>(ctx, m, 4.0);
            m->slice_state.store(2, std::memory_order_release);
            SPL_REQUIRE(ok, SPL_ERR_UNSUPPORTED, "sliced copy not built: padding above 4x or out of memory");
        }
        if (a->dtype == SPL_F32) spmv_sliced<float>(ctx, a, XLocal<float>{(const float *)x}, (float *)y);
        else spmv_sliced<double>(ctx, a, XLocal<double>{(const double *)x}, (double *)y);
        return;
    }
    if (kernel == SPL_SPMV_VECTOR) {
        if (a->dtype == SPL_F32) spmv_vector<float>(ctx, a, XLocal<float>{(const float *)x}, (float *)y, lanes, 0, a->nrows);
        else spmv_vector<double>(ctx, a, XLocal<double>{(const double *)x}, (double *)y, lanes, 0, a->nrows);
        return;
    }
    if (kernel == SPL_SPMV_MERGE) {
        spmv_plan(ctx, const_cast<spl_mat *>(a));
        if (a->dtype == SPL_F32) spmv_merge<float>(ctx, a, (const float *)x, (float *)y);
        else spmv_merge<double>(ctx, a, (const double *)x, (double *)y);
        return;
    }
    if (kernel == SPL_SPMV_SPLIT) {
        spl_mat *m = const_cast<spl_mat *>(a);
        spmv_plan(ctx, m);
        // The hot-column cache costs a histogram, a sort of the columns and a second index array
        // (~5 products' worth on the R-MAT matrix): it is built when a matrix comes back for its
        // second product, not for a one-off.
        if (m->hot_state.load(std::memory_order_acquire) != 2) {
            std::lock_guard<std::mutex> lock(m->plan_mu);
            const int st = m->hot_state.load(std::memory_order_relaxed);
            if (st == 0) {
                m->hot_state.store(1, std::memory_order_release);
            } else if (st == 1) {
                plan_hot_columns(ctx, m);
                SPL_CUDA(cudaStreamSynchronize(ctx->stream));
                m->hot_state.store(2, std::memory_order_release);
            }
        }
        if (a->dtype == SPL_F32) spmv_split<float>(ctx, a, (const float *)x, (float *)y);
        else spmv_split<double>(ctx, a, (const double *)x, (double *)y);
        return;
    }
    throw Error{SPL_ERR_UNSUPPORTED, "unknown SpMV kernel"};
}

// ------------------------------------------------------------------ host vectors, pipelined
// The reference-facing product takes x from host memory and returns y there.  Done as upload,
// product, download it is PCIe time twice over with the kernel in between; but a row chunk only
// needs the prefix of x up to its largest column, and its part of y can leave while the next chunk
// runs.  So x goes up in the prefixes the chunks need (stencils, bands: about a chunk's worth each;
// random columns: everything before the first chunk), the vector kernel runs chunk by chunk on the
// compute stream behind the upload events, and each chunk of y is copied down on a third stream
// behind the chunk's event: both directions of the link are busy at once.
namespace {

__global__ void chunk_need_kernel(const uint32_t *__restrict__ ptr, const uint32_t *__restrict__ ind, uint32_t nrows,
                                  uint32_t rows_per_chunk, uint32_t *__restrict__ need) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t m = 0;                                     // 1 + last (= largest) column of the row, 0 if empty
    if (r < nrows) {
        const uint32_t lo = ptr[r], hi = ptr[r + 1];
        if (hi > lo) m = ind[hi - 1] + 1u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    // rows_per_chunk is a multiple of 32: a warp never straddles two chunks
    if (lane_id() == 0 && m && r < nrows) atomicMax(need + (uint32_t)(r / rows_per_chunk), m);
}

void plan_pipeline(spl_ctx *ctx, spl_mat *a) {
    constexpr int K = spl_ctx::kPipeChunks;
    std::lock_guard<std::mutex> lock(a->plan_mu);
    if (a->pipe_state.load(std::memory_order_relaxed)) return;
    const uint32_t per = (uint32_t)((((uint64_t)a->nrows + K - 1) / K + 255) / 256 * 256);
    for (int c = 0; c <= K; ++c) a->pipe_rows[c] = (uint32_t)std::min<uint64_t>((uint64_t)c * per, a->nrows);
    uint32_t need[K] = {};
    SPL_CUDA(cudaMemsetAsync(ctx->d_scratch, 0, K * sizeof(uint32_t), ctx->stream));
    chunk_need_kernel<<<div_up(a->nrows, 256), 256, 0, ctx->stream>>>(a->ptr, a->ind, a->nrows, per, ctx->d_scratch);
    check_launch(ctx, "chunk_need");
    read_back(ctx, ctx->d_scratch, need, K);
    uint32_t run = 0;
    for (int c = 0; c < K; ++c) {                        // prefix maximum: what has to be up before chunk c runs
        run = std::max(run, need[c]);
        a->pipe_need[c] = run;
    }
    a->pipe_state.store(1, std::memory_order_release);
}

// The upload and download streams of the host-vector products and the events that order them against the compute
// stream, created on first use.
void pipe_streams(spl_ctx *ctx) {
    if (ctx->up_stream) return;
    SPL_CUDA(cudaStreamCreateWithFlags(&ctx->up_stream, cudaStreamNonBlocking));
    SPL_CUDA(cudaStreamCreateWithFlags(&ctx->down_stream, cudaStreamNonBlocking));
    for (cudaEvent_t &e : ctx->pipe_ev) SPL_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
}

// Pageable host memory makes every cudaMemcpyAsync block the host: copies overlap only with pinned memory.
bool is_pinned(const void *p) {
    cudaPointerAttributes at{};
    const bool ok = cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    return ok;
}

}  // namespace

bool spmv_host_pipelined(spl_ctx *ctx, const spl_mat *a, const void *x_host, void *y_host, void *x_dev,
                         void *y_dev) {
    constexpr int K = spl_ctx::kPipeChunks;
    a = csr_form(ctx, a);
    const size_t vs = a->vsize();
    if ((size_t)a->nrows * vs < (1u << 20) || a->nnz == 0) return false;      // small: one copy each way
    if (!is_pinned(x_host) || !is_pinned(y_host)) return false;               // nothing would overlap
    spl_mat *m = const_cast<spl_mat *>(a);
    spmv_plan(ctx, m);
    if (a->plan_kernel != SPL_SPMV_VECTOR) return false;                      // skewed rows: whole-matrix kernels
    if (!a->pipe_state.load(std::memory_order_acquire)) plan_pipeline(ctx, m);
    pipe_streams(ctx);
    cudaEvent_t *up_ev = ctx->pipe_ev, *run_ev = ctx->pipe_ev + K;
    cudaEvent_t start_ev = ctx->pipe_ev[2 * K], end_ev = ctx->pipe_ev[2 * K + 1];
    const unsigned char *xh = static_cast<const unsigned char *>(x_host);
    unsigned char *yh = static_cast<unsigned char *>(y_host);
    unsigned char *xd = static_cast<unsigned char *>(x_dev), *yd = static_cast<unsigned char *>(y_dev);
    // the device buffers were allocated in compute-stream order: the copy streams start behind that point
    SPL_CUDA(cudaEventRecord(start_ev, ctx->stream));
    SPL_CUDA(cudaStreamWaitEvent(ctx->up_stream, start_ev, 0));
    SPL_CUDA(cudaStreamWaitEvent(ctx->down_stream, start_ev, 0));
    uint32_t up = 0;
    for (int c = 0; c < K; ++c) {
        const uint32_t r0 = a->pipe_rows[c], r1 = a->pipe_rows[c + 1];
        if (r1 <= r0) continue;
        const uint32_t need = std::min(a->pipe_need[c], a->ncols);
        if (need > up) {
            SPL_CUDA(cudaMemcpyAsync(xd + (size_t)up * vs, xh + (size_t)up * vs, (size_t)(need - up) * vs,
                                     cudaMemcpyHostToDevice, ctx->up_stream));
            up = need;
        }
        SPL_CUDA(cudaEventRecord(up_ev[c], ctx->up_stream));
        SPL_CUDA(cudaStreamWaitEvent(ctx->stream, up_ev[c], 0));
        if (a->dtype == SPL_F32)
            spmv_vector<float>(ctx, a, XLocal<float>{(const float *)x_dev}, (float *)y_dev, a->plan_lanes, r0, r1);
        else
            spmv_vector<double>(ctx, a, XLocal<double>{(const double *)x_dev}, (double *)y_dev, a->plan_lanes, r0, r1);
        SPL_CUDA(cudaEventRecord(run_ev[c], ctx->stream));
        SPL_CUDA(cudaStreamWaitEvent(ctx->down_stream, run_ev[c], 0));
        SPL_CUDA(cudaMemcpyAsync(yh + (size_t)r0 * vs, yd + (size_t)r0 * vs, (size_t)(r1 - r0) * vs,
                                 cudaMemcpyDeviceToHost, ctx->down_stream));
    }
    // the compute stream (which the caller synchronises, and on which the buffers are freed) ends
    // behind the last download
    SPL_CUDA(cudaEventRecord(end_ev, ctx->down_stream));
    SPL_CUDA(cudaStreamWaitEvent(ctx->stream, end_ev, 0));
    return true;
}

// y = A x with only a WINDOW of x present: x_window holds the columns [start, start + len).  The matrix's
// column footprint (plan: smallest and largest stored column) must lie inside it.  This is the product
// of a row shard whose halo has been copied next to the rank's own slice (peer_barrier_halo): the
// kernels run with a plain local gather, at the speed of the unsharded product.
void spmv_window(spl_ctx *ctx, const spl_mat *a, const void *x_window, uint64_t start, uint64_t len, void *y) {
    a = csr_form(ctx, a);
    spmv_plan(ctx, const_cast<spl_mat *>(a));
    SPL_REQUIRE(start + len <= a->ncols && len > 0, SPL_ERR_ARG, "window outside the columns of A");
    SPL_REQUIRE(a->nnz == 0 || (a->col_min >= start && (uint64_t)a->col_max < start + len), SPL_ERR_SHAPE,
                "the matrix has stored columns outside the window of x");
    const unsigned char *base = static_cast<const unsigned char *>(x_window) - start * a->vsize();
    spmv(ctx, a, base, y, SPL_SPMV_AUTO, 0, (uint32_t)start, (uint32_t)(start + len));
}

// The row-sharded `&A * &x` with HOST vectors (the reference-facing call on one rank of a sharded
// matrix): this rank's slice of x goes up in chunks on the upload stream into its peer-visible slice,
// the device barrier publishes it, then the product runs row chunk by row chunk on the compute stream
// with each chunk of y going down on the download stream while the next chunk runs.  The barrier is
// a real dependence (peers gather from the slice), so upload and product do not overlap inside one
// step; product and download do.
void spmv_peer_host(spl_ctx *ctx, const spl_mat *a, const PeerX &px, void *const *flag_ptrs, uint32_t epoch,
                    uint32_t timeout_ms, const void *x_host_local, void *y_host_local, void *y_dev) {
    constexpr int K = spl_ctx::kPipeChunks;
    SPL_REQUIRE(a->format == SPL_CSR, SPL_ERR_UNSUPPORTED, "spl_spmv_peer_host needs a CSR matrix");
    spl_mat *m = const_cast<spl_mat *>(a);
    spmv_plan(ctx, m);
    const size_t vs = a->vsize();
    const uint32_t my_len = px.start[px.rank + 1] - px.start[px.rank];
    unsigned char *x_slice = static_cast<unsigned char *>(const_cast<void *>(px.slice[px.rank]));
    pipe_streams(ctx);
    cudaEvent_t *run_ev = ctx->pipe_ev + K;
    cudaEvent_t start_ev = ctx->pipe_ev[2 * K], end_ev = ctx->pipe_ev[2 * K + 1], up_ev = ctx->pipe_ev[0];
    // upload behind whatever the compute stream did to the slice before (a previous product may still gather from
    // the OTHER buffer; this one is free: see PeerVector)
    SPL_CUDA(cudaEventRecord(start_ev, ctx->stream));
    SPL_CUDA(cudaStreamWaitEvent(ctx->up_stream, start_ev, 0));
    SPL_CUDA(cudaStreamWaitEvent(ctx->down_stream, start_ev, 0));
    if (my_len)
        SPL_CUDA(cudaMemcpyAsync(x_slice, x_host_local, (size_t)my_len * vs, cudaMemcpyHostToDevice, ctx->up_stream));
    SPL_CUDA(cudaEventRecord(up_ev, ctx->up_stream));
    SPL_CUDA(cudaStreamWaitEvent(ctx->stream, up_ev, 0));
    peer_barrier(ctx, px.world, px.rank, flag_ptrs, epoch, timeout_ms);
    const int chunks = (is_pinned(y_host_local) && (size_t)a->nrows * vs >= (1u << 20)) ? K : 1;
    const uint32_t per = (uint32_t)((((uint64_t)a->nrows + chunks - 1) / chunks + 255) / 256 * 256);
    unsigned char *yd = static_cast<unsigned char *>(y_dev), *yh = static_cast<unsigned char *>(y_host_local);
    for (int c = 0; c < chunks; ++c) {
        const uint32_t r0 = (uint32_t)std::min<uint64_t>((uint64_t)c * per, a->nrows);
        const uint32_t r1 = (uint32_t)std::min<uint64_t>((uint64_t)(c + 1) * per, a->nrows);
        if (r1 <= r0) continue;
        if (a->dtype == SPL_F32) spmv_vector<float>(ctx, a, make_xpeer<float>(ctx, px), (float *)y_dev, a->plan_lanes, r0, r1);
        else spmv_vector<double>(ctx, a, make_xpeer<double>(ctx, px), (double *)y_dev, a->plan_lanes, r0, r1);
        SPL_CUDA(cudaEventRecord(run_ev[c], ctx->stream));
        SPL_CUDA(cudaStreamWaitEvent(ctx->down_stream, run_ev[c], 0));
        SPL_CUDA(cudaMemcpyAsync(yh + (size_t)r0 * vs, yd + (size_t)r0 * vs, (size_t)(r1 - r0) * vs,
                                 cudaMemcpyDeviceToHost, ctx->down_stream));
    }
    SPL_CUDA(cudaEventRecord(end_ev, ctx->down_stream));
    SPL_CUDA(cudaStreamWaitEvent(ctx->stream, end_ev, 0));
}

// Row-sharded SpMV with x left in its owners' memory (SURVEY.md 8e): the vector kernel with the
// peer gather.  Skewed shards should all-gather x and use the merge kernel instead.
void spmv_peer(spl_ctx *ctx, const spl_mat *a, const PeerX &px, void *y) {
    SPL_REQUIRE(a->format == SPL_CSR, SPL_ERR_UNSUPPORTED, "spl_spmv_peer needs a CSR matrix");
    spmv_plan(ctx, const_cast<spl_mat *>(a));
    if (a->dtype == SPL_F32) spmv_peer_t<float>(ctx, a, px, (float *)y, a->plan_lanes);
    else spmv_peer_t<double>(ctx, a, px, (double *)y, a->plan_lanes);
}

}  // namespace spl
