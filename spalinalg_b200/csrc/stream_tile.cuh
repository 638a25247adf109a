// stream_tile.cuh — the shared-memory tile of the stream SpMV kernels (spmv_stream_kernel in spmv.cu,
// spmv_gather_fused_kernel in gather.cu) and the row loop of their consumer warps.
//
// A tile is R = TILE_CONSUMERS / LPR consecutive rows: LPR lanes per row.  Its stored entries are one contiguous
// slice [lo, hi) of the CSR arrays; a producer copies the 16-byte aligned superset [slice_lo(lo), slice_hi(hi)) of
// the indices and values into a stage (the arrays carry slack behind their last entry), plus the row pointers of the
// tile in tile_ptr_slots(R) slots (R + 1 needed, whole 16-byte units).  A consumer finds its row's entries at stage
// positions [ptr[rl] - slice_lo(ptr[0]), ptr[rl + 1] - slice_lo(ptr[0])).
#pragma once

#include <cstdint>

namespace spl {

constexpr uint32_t TILE_CONSUMERS = 256;      // consumer threads of a CTA

__host__ __device__ constexpr uint32_t tile_rows(int lanes_per_row) { return TILE_CONSUMERS / (uint32_t)lanes_per_row; }
__host__ __device__ constexpr uint32_t tile_ptr_slots(uint32_t rows) { return rows + 4; }
__host__ __device__ constexpr uint32_t slice_lo(uint32_t lo) { return lo & ~3u; }
__host__ __device__ constexpr uint32_t slice_hi(uint32_t hi) { return (hi + 3u) & ~3u; }
// entries a stage holds when no window of a tile's rows holds more than `max_window`: the aligned superset of the
// largest slice
constexpr uint32_t stage_capacity(uint32_t max_window) { return (max_window + 6u + 3u) & ~3u; }

// acc += the row's products over stage positions [p0, e): lane `sub` of LPR takes positions p0 + sub, p0 + sub + LPR,
// ..., U of them in flight (all columns, then all U gathers of x, then the values).  Position j holds column
// cols[j] + cadd and value vals(j) (an array read, or a dictionary read through a one-byte code); gather(c) returns
// x[c].  A masked slot adds an explicit 0, never 0 * x (x may hold an inf).  These lines fix the bits of y: the
// vector kernel takes a row's entries in the same lane order.
template <typename T, int LPR, int U, typename V, typename G>
__device__ __forceinline__ void tile_row_sum(T &acc, const uint32_t *cols, uint32_t cadd, V vals, uint32_t p0,
                                             uint32_t e, uint32_t sub, G gather) {
    for (uint32_t j = p0 + sub; j < e; j += U * LPR) {
        uint32_t c[U];
        T xv[U], v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) c[u] = j + u * LPR < e ? cols[j + u * LPR] + cadd : 0xffffffffu;
#pragma unroll
        for (int u = 0; u < U; ++u) xv[u] = c[u] != 0xffffffffu ? gather(c[u]) : (T)0;
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = j + u * LPR < e ? vals(j + u * LPR) : (T)0;
#pragma unroll
        for (int u = 0; u < U; ++u) acc += j + u * LPR < e ? v[u] * xv[u] : (T)0;      // 0, never 0 * inf
    }
}

// Sum of acc over the LPR consecutive lanes of a row (every lane of the warp takes part).
template <int LPR, typename T>
__device__ __forceinline__ T row_lanes_sum(T acc) {
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return acc;
}

}  // namespace spl
