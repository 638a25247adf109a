// kernels.cuh — host-side entry points of each subsystem (one .cu file each); api.cu is the
// only caller.  Everything runs on ctx->stream; functions throw spl::Error.
#pragma once

#include "common.cuh"

namespace spl {

// assemble.cu — COO -> CSR/CSC (a-2, a-3, a-11 of SURVEY.md section 8)
spl_mat *assemble_from_coo_dev(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols,
                               uint32_t len, const uint32_t *row, const uint32_t *col,
                               const void *val, int dedup, int dropzero);
// wide_assemble.cu — the assembly entry of every COO front (spl_mat_from_coo{,_dev}, the builder):
// lists below 2^32 - 65536 triplets go to assemble_from_coo_dev unchanged; longer ones (or longer than
// SPL_ASSEMBLE_BUCKET_MAX when that is set) are assembled in buckets of whole majors, and the result is
// wide when it keeps 2^32 - 65536 entries or more.
bool assemble_is_bucketed(uint64_t len);
spl_mat *assemble_from_coo_any(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols,
                               uint64_t len, const uint32_t *row, const uint32_t *col,
                               const void *val, int dedup, int dropzero);
// Shared tail of assembly and SpGEMM: sorted (key = major << minor_bits | minor, value) records
// -> in-order segmented sum, optional zero drop, compaction, pointer array.  `vals` is updated
// in place.  key64 selects uint64 keys, else uint32.
spl_mat *finish_from_sorted(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols,
                            uint32_t n, bool key64, const void *keys, void *vals, int minor_bits,
                            int dedup, int dropzero);

// row-sharded assembly (8e): sender-side stable partition by owner, receiver-side assembly
void route_coo_dev(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols, uint32_t len,
                   const uint32_t *row, const uint32_t *col, const void *val, int world,
                   const uint64_t *major_starts, uint64_t *out_keys, void *out_val,
                   uint64_t *counts_host);
void route_count_dev(spl_ctx *ctx, int format, uint32_t nrows, uint32_t ncols, uint32_t len,
                     const uint32_t *row, const uint32_t *col, int world, const uint64_t *major_starts,
                     uint64_t *counts_host);
void route_coo_peers_dev(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols, uint32_t len,
                         const uint32_t *row, const uint32_t *col, const void *val, int world,
                         const uint64_t *major_starts, void *const *key_bufs, void *const *val_bufs,
                         const uint64_t *dst_offsets);
spl_mat *assemble_from_packed_dev(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols,
                                  uint32_t len, const uint64_t *keys, const void *val, int dedup,
                                  int dropzero);

// recompress.cu — transpose / CSR<->CSC (a-4, a-5): same entries grouped by the other index.
void recompress(spl_ctx *ctx, int dtype, uint32_t nmajor, uint32_t nminor, uint32_t nnz,
                const uint32_t *ptr, const uint32_t *ind, const void *val, uint32_t *out_ptr,
                uint32_t *out_ind, void *out_val);

// spmv.cu — y = A x (a-6 restricted to B = n x 1, dense vectors).  CSR runs the row kernels; a CSC
// matrix runs them on its cached CSR form (csr_form), or scatters column by column (SPL_SPMV_SCATTER).
void spmv_plan(spl_ctx *ctx, spl_mat *a);
// `a` itself if it is CSR, else its CSR twin (built on first use, kept with the matrix)
const spl_mat *csr_form(spl_ctx *ctx, const spl_mat *a);
// forget everything derived from the values (after values_mut): CSR twin, sliced copy
void drop_value_copies(spl_ctx *ctx, spl_mat *m);
void spmv(spl_ctx *ctx, const spl_mat *a, const void *x, void *y, int kernel, int lanes, uint32_t x_lo = 0,
          uint32_t x_hi = 0);
// y = A x where x_window holds only the columns [start, start + len) of x (the matrix's column footprint
// must lie inside): the product of a row shard next to its halo
void spmv_window(spl_ctx *ctx, const spl_mat *a, const void *x_window, uint64_t start, uint64_t len, void *y);
// `&A * &x` with host vectors, pipelined: x goes up in prefixes, row chunks run as soon as the prefix
// they need is there, their part of y goes down while the next chunk runs (PCIe both ways at once).
// x_dev / y_dev are device buffers of ncols / nrows values.  Returns false (nothing done) when the
// matrix is not one for the vector kernel or too small to be worth it; the caller then does the
// plain upload - product - download.  Does not synchronise the compute stream.
bool spmv_host_pipelined(spl_ctx *ctx, const spl_mat *a, const void *x_host, void *y_host, void *x_dev,
                         void *y_dev);

// x gathered from the slice that owns the column (local HBM or a peer's over NVLink)
struct PeerX {
    const void *slice[SPL_MAX_PEERS];
    uint32_t start[SPL_MAX_PEERS + 1];
    int world;
    int rank;
};
void spmv_peer(spl_ctx *ctx, const spl_mat *a, const PeerX &px, void *y);
// the same with this rank's slices of x and y in host memory: upload into the rank's peer slice,
// barrier, product in row chunks with the download of each chunk behind it (does not synchronise)
void spmv_peer_host(spl_ctx *ctx, const spl_mat *a, const PeerX &px, void *const *flag_ptrs, uint32_t epoch,
                    uint32_t timeout_ms, const void *x_host_local, void *y_host_local, void *y_dev);

// gather.cu — general shards: the all-gather of x fused into the product (one persistent kernel)
void spmv_gather_fused(spl_ctx *ctx, int dtype, uint32_t nloc, int world, int rank, const uint64_t *col_starts,
                       const void *const *x_slices, int nblocks, const uint32_t *block_first, const uint32_t *bptr,
                       uint32_t pstride, const uint32_t *tile_caps, const uint32_t *bind, const void *bval, void *x_full,
                       void *y, uint32_t *ready, uint32_t epoch, double entries_per_row, void *const *flag_ptrs,
                       uint32_t barrier_epoch, uint32_t timeout_ms, unsigned long long *timeline);

// peer.cu — CUDA IPC buffers and the flag barrier over peer memory
void peer_barrier(spl_ctx *ctx, int world, int rank, void *const *flag_ptrs, uint32_t epoch,
                  uint32_t timeout_ms);
void peer_pull(spl_ctx *ctx, int world, int rank, size_t vsize, const uint64_t *starts,
               const void *const *slices, void *x_full);
// the barrier, then this rank's halo: the halo_left columns before and the halo_right columns after its own
// slice are copied from their owners' slices into the padding around slices[rank] (one small kernel)
void peer_barrier_halo(spl_ctx *ctx, int world, int rank, void *const *flag_ptrs, uint32_t epoch, uint32_t timeout_ms,
                       size_t vsize, const uint64_t *starts, void *const *slices, uint32_t halo_left, uint32_t halo_right);

// addsub.cu — C = A +/- B on compressed arrays of equal format (a-7)
spl_mat *addsub(spl_ctx *ctx, const spl_mat *a, const spl_mat *b, int subtract);

// spgemm.cu — C = A * B (a-6): expand products in ascending-k order, stable sort, in-order sum
spl_mat *spgemm(spl_ctx *ctx, const spl_mat *a, const spl_mat *b);

// misc.cu
void negate(spl_ctx *ctx, int dtype, uint32_t nnz, const void *val, void *out);
// 0 = valid, else the reference assertion ordinal (7, 8 or 9); ptr[0] and ptr[n] are checked by
// the caller.
int validate_compressed(spl_ctx *ctx, uint32_t nmajor, uint32_t nminor, uint32_t nnz,
                        const uint32_t *ptr, const uint32_t *ind);
// dst[i] = (uint32) src[i]; returns (through d_flag != 0) whether any src[i] >= limit.
void narrow_u64(spl_ctx *ctx, const uint64_t *src, uint32_t *dst, size_t n, uint64_t limit,
                uint32_t *d_flag);
void widen_u32(spl_ctx *ctx, const uint32_t *src, uint64_t *dst, size_t n);
void fill_eye(spl_ctx *ctx, int dtype, uint32_t size, uint32_t *ptr, uint32_t *ind, void *val);
// major index of every stored entry (rowptr expansion, src/csr.rs:303-316)
void expand_major(spl_ctx *ctx, uint32_t nmajor, uint32_t nnz, const uint32_t *ptr, uint32_t *out);
// (major, minor) of the stored entries [start, start + count) as uint64 (the chunks of iter())
void entry_range(spl_ctx *ctx, const spl_mat *m, uint32_t start, uint32_t count, uint64_t *major_out,
                 uint64_t *minor_out);
// ptr[q] = first position p with sorted_major[p] >= q, for q in [0, nmajor]
void fill_ptr(spl_ctx *ctx, const uint32_t *sorted_major, uint32_t nnz, uint32_t nmajor,
              uint32_t *ptr);

spl_mat *new_mat(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols, uint32_t nnz);

// wide.cu — matrices with 2^32 - 65536 stored entries or more (64-bit positions, spl_mat::ptr64)
// Entry count from which a new matrix is stored wide: 2^32 - 65536, or SPL_WIDE_MIN_NNZ when that is set.
uint64_t wide_min_nnz();
spl_mat *new_wide_mat(spl_ctx *ctx, int format, int dtype, uint32_t nrows, uint32_t ncols, uint64_t nnz);
int wide_validate(spl_ctx *ctx, const spl_mat *m);      // 0, or the failing assertion of CsrMatrix::new (7, 8, 9)
void wide_spmv(spl_ctx *ctx, const spl_mat *a, const void *x, void *y);
spl_mat *wide_regroup(spl_ctx *ctx, const spl_mat *in, int out_format, uint32_t out_rows, uint32_t out_cols);
void wide_entry_range(spl_ctx *ctx, const spl_mat *m, uint64_t start, uint32_t count, uint64_t *major_out,
                      uint64_t *minor_out);
// out[i] = in[0] + ... + in[i - 1] for i in [0, n] (64-bit sums of 32-bit counts)
void wide_exclusive_scan(spl_ctx *ctx, const uint32_t *in, uint32_t n, uint64_t *out);
uint32_t wide_max_u32(spl_ctx *ctx, const uint32_t *a, uint32_t n);      // largest of a[0..n), 0 if n == 0
void free_mat(spl_ctx *ctx, spl_mat *m);

}  // namespace spl
