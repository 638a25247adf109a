/*
 * spl.h — C ABI of libspalinalg_b200.so: the B200 (sm_100a) implementation of
 * spalinalg's data-parallel sparse hot path.
 *
 * The reference (Rust crate spalinalg v0.0.2) has no FFI layer: its boundary is
 * the crate's public API reached by static trait dispatch (SURVEY.md 8b).  Each
 * entry point below names the reference item (file:line under /root/reference)
 * it stands in for; INTEGRATION.md shows the Rust `extern "C"` block and the
 * `impl From/Add/Sub/Mul/Neg` shims a maintainer would add on top.
 *
 * Conventions
 *  - Plain pointers and sizes only.  Host index arrays are uint64_t (Rust usize);
 *    device index arrays are uint32_t.  Values are float or double, selected by
 *    spl_dtype.  All matrices live in device memory behind an opaque spl_mat.
 *  - Every function returns an spl_status.  Nothing unwinds across the ABI; the
 *    Rust shim turns a non-zero status into panic!, the reference's convention
 *    (assert!/assert_eq!, e.g. src/csr.rs:144-156, src/csr/ops/add.rs:9-10).
 *  - One spl_ctx per host thread (it owns a stream and the last-error text).
 *    spl_mat objects are immutable after creation and may be shared read-only.
 *  - There is no CPU fallback: without a CUDA device spl_ctx_create fails.
 *  - Limits: dims below 2^32 (device indices are 32 bit).  Positions are 32 bit on the fast
 *    paths; a CsrMatrix / CscMatrix with 2^32 - 65536 stored entries or more ("wide") keeps a 64-bit
 *    pointer array on the device and supports construction + validation, SpMV (CSR only), transpose,
 *    CSR<->CSC, download and chunked iteration, and COO assembly produces it from 2^32 - 65536 triplets
 *    or more (fewer than that per row of a CSR, per column of a CSC result).  Add/sub/mul/neg,
 *    set_values, to_coo, the windowed and sharded products and SpMV of a wide CSC matrix answer
 *    SPL_ERR_UNSUPPORTED for it (their lengths and intermediate products stay below 2^32 - 65536).
 *    Test-only setting: the environment variable SPL_WIDE_MIN_NNZ=<n> makes every matrix created with
 *    n stored entries or more wide (n clamped to [1, 2^32 - 65536]; a value that is not a number is
 *    ignored; a matrix without entries is never wide), so that the wide kernels can be compared with
 *    the usual ones at small sizes.  It applies to spl_mat_from_compressed,
 *    spl_mat_from_compressed_dev64 and the result of bucketed COO assembly (see
 *    SPL_ASSEMBLE_BUCKET_MAX); transposes and conversions keep the width of their input.
 */
#ifndef SPL_H
#define SPL_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct spl_ctx spl_ctx;
typedef struct spl_mat spl_mat;

typedef enum {
    SPL_OK = 0,
    SPL_ERR_SHAPE = 1,       /* operand shapes disagree (assert_eq! on dims) */
    SPL_ERR_INVALID = 2,     /* CsrMatrix::new / CscMatrix::new would panic; see spl_invalid_reason */
    SPL_ERR_CUDA = 3,
    SPL_ERR_UNSUPPORTED = 4,
    SPL_ERR_OOM = 5,
    SPL_ERR_ARG = 6          /* NULL handle, unknown enum, index out of range in COO input */
} spl_status;

typedef enum { SPL_CSR = 0, SPL_CSC = 1 } spl_format;
typedef enum { SPL_F32 = 0, SPL_F64 = 1 } spl_dtype;   /* Scalar: src/scalar.rs:55-57 */

/* Row sharding across the GPUs of one box (SURVEY.md 8e): at most this many ranks. */
#define SPL_MAX_PEERS 8
#define SPL_IPC_HANDLE_BYTES 64

/* SpMV kernel choice (spl_spmv_ex): auto picks by row-length statistics — VECTOR (1..32 lanes per
 * row) for regular rows, SPLIT (fixed chunks of stored entries per warp, the merge-path balance at
 * warp granularity) for skewed rows; MERGE is the block-level merge-path kernel, selectable.  SLICED
 * is the lane-per-row kernel over a second copy of the matrix kept in slices of 32 rows, column-major
 * inside the slice (every load a full line; the row sum runs in ascending column order, i.e. it is
 * bit-identical to the reference's `&A * &X`); AUTO builds the copy for regular matrices when they
 * come back for a second product and the padding stays small.  STREAM is the persistent kernel for
 * regular rows: one producer thread per CTA moves the contiguous col/val slice of a tile of rows
 * into a ring of shared-memory stages with TMA bulk copies (cp.async.bulk + mbarrier) several tiles
 * ahead, the other warps consume the stages (x gathers, row sums with LPR lanes per row; with one
 * lane per row the sum runs in ascending column order, bit-identical to `&A * &X`).  Launched with
 * programmatic dependent launch: the matrix prefetch of a product overlaps the tail of the one before.
 * SCATTER is for CSC matrices only: column by column with atomic adds into y, no second copy of the
 * matrix (every other choice runs a CSC matrix on its cached CSR form, see spl_spmv). */
typedef enum { SPL_SPMV_AUTO = 0, SPL_SPMV_VECTOR = 1, SPL_SPMV_MERGE = 2, SPL_SPMV_SPLIT = 3, SPL_SPMV_SLICED = 4,
               SPL_SPMV_STREAM = 5, SPL_SPMV_SCATTER = 6 } spl_spmv_kernel;

/* ---- context ------------------------------------------------------------ */

/* device: CUDA ordinal.  stream: a cudaStream_t to run on (e.g. the caller's
 * current stream), or NULL to let the context create its own. */
int spl_ctx_create(int device, void *stream, spl_ctx **out);
int spl_ctx_destroy(spl_ctx *ctx);
int spl_ctx_sync(spl_ctx *ctx);
/* Synchronises, then returns the freed device memory that the library's own pool keeps for reuse to the
 * driver (matrices and builders that are alive are untouched).  For callers about to allocate most of
 * the device themselves. */
int spl_ctx_trim(spl_ctx *ctx);
/* Page-locked host memory for the vectors of spl_spmv_host / spl_spmv_peer_host: with pinned x and y the
 * upload, the product and the download are pipelined over row chunks; pageable vectors take one blocking
 * copy each way (the result is the same).  spl_host_alloc / spl_host_free allocate such memory;
 * spl_host_register / spl_host_unregister pin memory the caller already owns, in place (costs about as
 * much as copying it: once per buffer, not per product).  No context: SPL_OK, SPL_ERR_ARG or SPL_ERR_CUDA. */
int spl_host_alloc(uint64_t bytes, void **out);
int spl_host_free(void *p);
int spl_host_register(void *p, uint64_t bytes);
int spl_host_unregister(void *p);
const char *spl_last_error(const spl_ctx *ctx);
/* After SPL_ERR_INVALID: 1-based ordinal of the failing assertion of
 * CsrMatrix::new (src/csr.rs:144-156) / CscMatrix::new (src/csc.rs:144-156):
 * 1 nrows>0, 2 ncols>0, 3 ptr.len()==n+1, 4 ptr[0]==0, 5 ind.len()==ptr[n],
 * 6 values.len()==ptr[n], 7 ptr sorted, 8 index in range, 9 indices strictly
 * increasing inside a row/column. */
int spl_invalid_reason(const spl_ctx *ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t spl_launch_count(const spl_ctx *ctx);

/* ---- construction --------------------------------------------------------- */

/* COO -> CSR/CSC assembly.
 *   impl From<&CooMatrix<T>> for CsrMatrix<T>   src/csr/conv/coo.rs:3-116
 *   impl From<&CooMatrix<T>> for CscMatrix<T>   src/csc/conv/coo.rs:3-116
 * Entries sorted by (row, col) [(col, row) for CSC]; duplicates of a cell summed
 * sequentially in insertion order; sums == 0 dropped.  Bit-exact against the
 * reference in structure and values.  dedup=0, dropzero=0 gives
 *   impl From<&DokMatrix<T>> for CsrMatrix<T>   src/csr/conv/dok.rs:3-76
 *   impl From<&DokMatrix<T>> for CscMatrix<T>   src/csc/conv/dok.rs:3-76
 * (keys unique, explicit zeros kept).  Host SoA arrays of length len; the bound
 * checks of CooMatrix::push (src/coo.rs:431-435) are re-checked on the device
 * (SPL_ERR_ARG).  nrows, ncols must be > 0 (src/coo.rs:105-106).
 * len may be 2^32 - 65536 or more: the list is then assembled in buckets of whole rows (CSR) / columns
 * (CSC), each assembled as a shorter list and the parts stitched, with the same result bit for bit.  The
 * result is wide (64-bit pointers) when it keeps 2^32 - 65536 entries or more, else an ordinary matrix.
 * One row (CSR) / column (CSC) with 2^32 - 65536 triplets or more gives SPL_ERR_UNSUPPORTED.  Bucket size
 * follows the device memory free at the call; the peak is the input + one bucket's scratch (about
 * 3 (8 + V) bytes per triplet) + the parts so far, and at the end the input + the parts + the output.
 * The host front uploads such a list through a fixed staging buffer. */
int spl_mat_from_coo(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                     uint64_t len, const uint64_t *row, const uint64_t *col, const void *val,
                     int dedup, int dropzero, spl_mat **out);
/* Same with device-resident uint32 SoA input (inputs are not modified). */
int spl_mat_from_coo_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                         uint64_t len, const uint32_t *row_dev, const uint32_t *col_dev,
                         const void *val_dev, int dedup, int dropzero, spl_mat **out);

/* ---- CooMatrix storage that streams to the device while it is filled (SURVEY.md 8f-4) ----
 * spl_coo is the storage of a CooMatrix<T> (src/coo.rs:52-57): insertion-ordered triplets kept as
 * three PINNED host arrays (row usize, col usize, value).  Every time another 2^19 triplets are
 * complete they are sent on the builder's own copy stream (indices narrowed to uint32 on the
 * device), so the host keeps pushing while the DMA engine works and the conversion finds its input
 * already in HBM.  One builder per host thread at a time (`&mut self` in the reference).
 *   spl_coo_create    CooMatrix::new / with_capacity   src/coo.rs:104-112, 162-170
 *   spl_coo_push      CooMatrix::push                  src/coo.rs:431-435 (bounds -> SPL_ERR_ARG)
 *   spl_coo_extend    Extend for CooMatrix             src/coo.rs:566-573 (all entries asserted
 *                                                      before any is stored); with_triplets :254-288
 *   spl_coo_truncate  pop / clear                      src/coo.rs:450-452, 470-472
 *   spl_coo_len / _capacity                            src/coo.rs:349-351, 366-368
 *   spl_coo_host_ptrs get / iter (borrowed, valid until the next push/extend/reserve)
 *                                                      src/coo.rs:386-390, 491-495
 *   spl_coo_invalidate get_mut / iter_mut                src/coo.rs:408-412, 514-518: the caller is about to
 *                     write values through the host pointers from entry `first` on; what the copy
 *                     stream already took from there is sent again at the next conversion
 *   spl_mat_from_coo_builder   From<&CooMatrix> for CsrMatrix / CscMatrix (as spl_mat_from_coo, any
 *                     length); the builder stays valid and can be pushed to and converted again. */
typedef struct spl_coo spl_coo;
int spl_coo_create(spl_ctx *ctx, int dtype, uint64_t nrows, uint64_t ncols, uint64_t capacity,
                   spl_coo **out);
int spl_coo_free(spl_coo *coo);
const char *spl_coo_last_error(const spl_coo *coo);
int spl_coo_push(spl_coo *coo, uint64_t row, uint64_t col, const void *value);
int spl_coo_extend(spl_coo *coo, uint64_t len, const uint64_t *row, const uint64_t *col, const void *val);
int spl_coo_reserve(spl_coo *coo, uint64_t capacity);
int spl_coo_truncate(spl_coo *coo, uint64_t len);
uint64_t spl_coo_len(const spl_coo *coo);
uint64_t spl_coo_capacity(const spl_coo *coo);
/* Entries already handed to the copy stream (diagnostic). */
uint64_t spl_coo_streamed(const spl_coo *coo);
int spl_coo_invalidate(spl_coo *coo, uint64_t first);
int spl_coo_host_ptrs(const spl_coo *coo, const uint64_t **row, const uint64_t **col, const void **val);
int spl_mat_from_coo_builder(spl_ctx *ctx, spl_coo *coo, int format, int dedup, int dropzero,
                             spl_mat **out);

/* CsrMatrix::new (src/csr.rs:137-164) / CscMatrix::new (src/csc.rs:137-164):
 * validating constructor from host arrays.  ptr is rowptr (CSR) or colptr (CSC). */
int spl_mat_from_compressed(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                            uint64_t ptr_len, const uint64_t *ptr,
                            uint64_t ind_len, const uint64_t *ind,
                            uint64_t val_len, const void *val, spl_mat **out);
/* Same from device uint32 arrays (copied); validate=0 skips the checks. */
int spl_mat_from_compressed_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                                uint64_t nnz, const uint32_t *ptr_dev, const uint32_t *ind_dev,
                                const void *val_dev, int validate, spl_mat **out);
/* The same with a 64-bit device pointer array (usize, src/csr.rs:66-72): the constructor for matrices
 * with 2^32 - 65536 stored entries or more, which stay "wide" (64-bit positions) on the device; smaller
 * ones are narrowed to the usual form. */
int spl_mat_from_compressed_dev64(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                                  uint64_t nnz, const uint64_t *ptr_dev, const uint32_t *ind_dev,
                                  const void *val_dev, int validate, spl_mat **out);
/* CsrMatrix::eye (src/csr.rs:179-188) / CscMatrix::eye (src/csc.rs:179-188). */
int spl_mat_eye(spl_ctx *ctx, int format, int dtype, uint64_t size, spl_mat **out);

/* ---- the hot path --------------------------------------------------------- */

/* From<&CsrMatrix> for CscMatrix (src/csc/conv/csr.rs:3-53) and
 * From<&CscMatrix> for CsrMatrix (src/csr/conv/csc.rs:3-53): same matrix, other
 * format.  format == the input's format yields a copy. */
int spl_mat_convert(spl_ctx *ctx, const spl_mat *in, int format, spl_mat **out);
/* CsrMatrix::transpose (src/csr.rs:358-406), CscMatrix::transpose (src/csc.rs:358-406). */
int spl_mat_transpose(spl_ctx *ctx, const spl_mat *in, spl_mat **out);
/* impl Add / Sub for &CsrMatrix (src/csr/ops/add.rs:5-75, sub.rs:5-75) and
 * &CscMatrix (src/csc/ops/add.rs:5-70, sub.rs:5-70).  Pattern union, explicit
 * zeros kept, one IEEE op per overlap: bit-exact. */
int spl_mat_add(spl_ctx *ctx, const spl_mat *a, const spl_mat *b, spl_mat **out);
int spl_mat_sub(spl_ctx *ctx, const spl_mat *a, const spl_mat *b, spl_mat **out);
/* impl Mul for &CsrMatrix (src/csr/ops/mul.rs:5-60) / &CscMatrix
 * (src/csc/ops/mul.rs:5-61): C = A*B, each C[i,j] accumulated over ascending k
 * with the product rounded before the add; structural union, no zero drop. */
int spl_mat_mul(spl_ctx *ctx, const spl_mat *a, const spl_mat *b, spl_mat **out);
/* impl Neg (src/csr/ops/neg.rs:5-18, src/csc/ops/neg.rs:5-18). */
int spl_mat_neg(spl_ctx *ctx, const spl_mat *a, spl_mat **out);

/* y = A*x with dense device vectors (extension; the reference's only route is
 * `&A * &X` with X n x 1, src/csr/ops/mul.rs:5-60 and src/csc/ops/mul.rs:5-61, whose values
 * this matches to 1e-12 (f64) / 1e-5 (f32) relative; rows without entries give 0).  x has
 * ncols elements, y nrows.  A may be CSR or CSC: the first product on a CSC matrix builds
 * its CSR form on the device (as spl_mat_convert would) and keeps it with the matrix, so
 * later products cost the same as on a CsrMatrix.  With A = the CSC view of a CSR matrix B
 * (same arrays, dims swapped) this is y = B^T x. */
int spl_spmv(spl_ctx *ctx, const spl_mat *a, const void *x_dev, void *y_dev);
/* kernel: spl_spmv_kernel in bits 0-7; bits 8-15 optionally force the vector kernel's lanes per
 * row (1, 2, 4, 8, 16 or 32; 0 = planned value).  On a wide matrix the argument is ignored: every
 * value runs the vector kernel with 64-bit positions and lanes chosen from the mean row length, and
 * gives the same bytes.  A wide matrix must be CSR: a wide CSC one gives SPL_ERR_UNSUPPORTED (convert
 * it with spl_mat_convert first). */
int spl_spmv_ex(spl_ctx *ctx, const spl_mat *a, const void *x_dev, void *y_dev, int kernel);
/* Host-buffer form (the reference-facing `&A * &x`): uploads x, runs spl_spmv, downloads y,
 * synchronises.  With pinned vectors of a megabyte or more and a matrix for the vector kernel the
 * three steps are pipelined over row chunks (x in the prefixes the chunks need, y chunk by chunk
 * behind the kernels), so both directions of the PCIe link work at once; same result bit for bit. */
int spl_spmv_host(spl_ctx *ctx, const spl_mat *a, const void *x_host, void *y_host);
/* Which kernel AUTO resolves to for this matrix (SPL_SPMV_VECTOR / _SPLIT) and the vector kernel's
 * lanes per row.  A wide matrix answers SPL_SPMV_VECTOR and 0 lanes (its kernel picks the lanes at
 * each product). */
int spl_spmv_choice(spl_ctx *ctx, const spl_mat *a, int *kernel, int *lanes_per_row);

/* ---- access --------------------------------------------------------------- */

/* nrows/ncols/nnz accessors (src/csr.rs:200-289). Any out pointer may be NULL. */
int spl_mat_info(const spl_mat *m, int *format, int *dtype, uint64_t *nrows, uint64_t *ncols,
                 uint64_t *nnz);
/* rowptr()/colind()/values() (src/csr.rs:228-258) as host copies, indices widened
 * to usize.  ptr needs nmajor+1 slots, ind and val nnz.  Synchronises. */
int spl_mat_download(spl_ctx *ctx, const spl_mat *m, uint64_t *ptr, uint64_t *ind, void *val);
/* values_mut() (src/csr.rs:270-272, src/csc.rs:270-272): overwrite the stored values, structure
 * kept.  val points to nnz host values of the matrix's scalar type.  Needs exclusive access to the
 * matrix, as `&mut self` does in the reference. */
int spl_mat_set_values(spl_ctx *ctx, spl_mat *m, const void *val);
/* Borrow the device arrays (uint32 ptr[nmajor+1], uint32 ind[nnz], T val[nnz]). */
int spl_mat_device_ptrs(const spl_mat *m, const uint32_t **ptr_dev, const uint32_t **ind_dev,
                        const void **val_dev);
/* The 64-bit pointer array of a wide matrix (NULL for the usual ones, whose spl_mat_device_ptrs ptr is
 * then valid instead). */
int spl_mat_device_ptr64(const spl_mat *m, const uint64_t **ptr64_dev);
/* From<&CsrMatrix>/<&CscMatrix> for CooMatrix (src/coo.rs:629-705): expand to
 * host triplets in storage order.  Arrays need nnz slots.  Synchronises. */
int spl_mat_to_coo(spl_ctx *ctx, const spl_mat *m, uint64_t *row, uint64_t *col, void *val);
/* The same conversion with the result left in device memory (uint32 SoA triplets, nnz slots each):
 * the input format of spl_mat_from_coo_dev / spl_coo_route_dev, so results flow back into the builder
 * format without visiting the host (SURVEY.md 8f-2).  Asynchronous on the context's stream. */
int spl_mat_to_coo_dev(spl_ctx *ctx, const spl_mat *m, uint32_t *row_dev, uint32_t *col_dev, void *val_dev);
/* iter() / into_iter() on a device-resident matrix (src/csr.rs:303-316, 409-440; src/csc.rs same
 * lines): the stored entries [start, start + count) in storage order as host triplets.  An iterator
 * reads the matrix chunk by chunk through this call instead of materialising nnz tuples at once; the
 * row (column) of an entry is found from the pointer array on the device.  Synchronises. */
int spl_mat_read_entries(spl_ctx *ctx, const spl_mat *m, uint64_t start, uint64_t count, uint64_t *row,
                         uint64_t *col, void *val);
int spl_mat_free(spl_ctx *ctx, spl_mat *m);

/* ---- row sharding across GPUs (one process per GPU; SURVEY.md 8e) ----------------
 * The reference is single-process; these entry points are the sharded forms of the
 * same reference items.  Rank g owns the contiguous block [starts[g], starts[g+1]) of
 * the major axis (rows for CSR).  Collectives that move bulk data (the all-to-all of
 * routed triplets, the all-gather of x for general matrices) stay with the caller's
 * communicator (NCCL through torch.distributed); what is declared here is the device
 * work either side of them and the peer-memory path that needs no collective. */

/* Sending side of sharded From<&CooMatrix> (src/csr/conv/coo.rs:3-116,
 * src/csc/conv/coo.rs:3-116): stable partition of this rank's triplets by owning
 * rank.  keys_out_dev[i] = (major - starts[owner]) << bits(nminor) | minor, bits(n) =
 * ceil(log2 n); vals_out_dev carries the values; both have len slots and hold the
 * share of rank 0 first, then rank 1, ...; counts_host[g] = entries for rank g.
 * Inside a share the insertion order is kept, so concatenating the received shares in
 * source-rank order keeps the global insertion order among duplicates. */
int spl_coo_route_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                      uint64_t len, const uint32_t *row_dev, const uint32_t *col_dev,
                      const void *val_dev, int world, const uint64_t *major_starts,
                      uint64_t *keys_out_dev, void *vals_out_dev, uint64_t *counts_host);
/* The same routing fused with the exchange, over peer memory (no staging buffer, no all-to-all):
 * spl_coo_route_count_dev checks the bounds and counts this rank's triplets per owning rank; the
 * caller shares the counts, sizes the receive buffers (spl_peer_alloc / spl_peer_open) and gives
 * every sender its slot: dst_offsets[g] = entries that ranks before this one send to rank g.
 * spl_coo_route_peers_dev then runs the stable partition and writes each record straight into its
 * owner's buffers key_bufs[g] (uint64 packed keys) / val_bufs[g] over NVLink.  Bracket it with
 * spl_peer_barrier: before (the owners are done with the previous contents) and after (every
 * record has landed). */
int spl_coo_route_count_dev(spl_ctx *ctx, int format, uint64_t nrows, uint64_t ncols, uint64_t len,
                            const uint32_t *row_dev, const uint32_t *col_dev, int world,
                            const uint64_t *major_starts, uint64_t *counts_host);
int spl_coo_route_peers_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                            uint64_t len, const uint32_t *row_dev, const uint32_t *col_dev,
                            const void *val_dev, int world, const uint64_t *major_starts,
                            void *const *key_bufs, void *const *val_bufs, const uint64_t *dst_offsets);
/* Receiving side: assembly of one shard (nrows x ncols are the SHARD's dimensions)
 * from packed keys as produced by spl_coo_route_dev.  Same semantics and bit-exactness
 * as spl_mat_from_coo_dev. */
int spl_mat_from_packed_dev(spl_ctx *ctx, int format, int dtype, uint64_t nrows, uint64_t ncols,
                            uint64_t len, const uint64_t *keys_dev, const void *vals_dev,
                            int dedup, int dropzero, spl_mat **out);

/* Peer-visible device memory (CUDA IPC over NVLink/NVSwitch).  alloc returns a zeroed
 * cudaMalloc block plus the handle to send to the other ranks; open maps a peer's block
 * into this process (peer access is enabled on demand). */
int spl_peer_alloc(spl_ctx *ctx, uint64_t bytes, void **dev_ptr, unsigned char *handle_out);
int spl_peer_open(spl_ctx *ctx, const unsigned char *handle, void **peer_ptr);
int spl_peer_close(spl_ctx *ctx, void *peer_ptr);
int spl_peer_free(spl_ctx *ctx, void *dev_ptr);
/* Device-side barrier over peer memory: flag_ptrs[g] is rank g's uint32[SPL_MAX_PEERS]
 * flag block (own block included, all zero-initialised); epoch must grow by one per
 * call on every rank.  Everything this rank's stream wrote before the barrier is
 * visible to peers' kernels launched after it.  Bounded spin: SPL_ERR_CUDA after
 * timeout_ms if a peer never arrives (reported at the next synchronising call through
 * spl_peer_barrier_status). */
int spl_peer_barrier(spl_ctx *ctx, int world, int rank, void *const *flag_ptrs, uint32_t epoch,
                     uint32_t timeout_ms);
int spl_peer_barrier_status(spl_ctx *ctx, int *timed_out);
/* Barrier + halo for banded / stencil shards whose slices are allocated with padding: after the
 * barrier (same protocol and arguments as spl_peer_barrier), the halo_left columns before and the
 * halo_right columns after this rank's own slice are copied from their owners' slices x_slices[g]
 * (= &x[starts[g]]) into the memory just before / after x_slices[rank], which the caller allocated
 * with that much room (halo_left * V bytes before the slice, halo_right * V after).  One launch; the
 * product that follows (spl_spmv_window) reads one local array. */
int spl_peer_barrier_halo(spl_ctx *ctx, int world, int rank, void *const *flag_ptrs, uint32_t epoch,
                          uint32_t timeout_ms, int dtype, const uint64_t *starts, void *const *x_slices,
                          uint64_t halo_left, uint64_t halo_right);
/* y = A*x where only the columns [window_start, window_start + window_len) of x are present, at
 * x_window_dev (x_window_dev[0] = x[window_start]).  Every stored column of A must lie in the window
 * (SPL_ERR_SHAPE otherwise): the row shard of a banded / stencil matrix beside its halo.  Same
 * kernels and results as spl_spmv. */
int spl_spmv_window(spl_ctx *ctx, const spl_mat *a, const void *x_window_dev, uint64_t window_start,
                    uint64_t window_len, void *y_dev);
/* Smallest and largest stored column of A (0, 0 for an empty matrix): sizes the halo. */
int spl_spmv_footprint(spl_ctx *ctx, const spl_mat *a, uint64_t *col_min, uint64_t *col_max);
/* All-gather of x by pulling over peer memory, for general (random / power-law) shards whose
 * gathers would be 4-byte NVLink transactions: one kernel copies every peer's slice
 * (slices[g] = x[starts[g] .. starts[g+1]), mapped with spl_peer_open) into the local full-length
 * vector x_full_dev with TMA bulk copies through a shared-memory ring (one thread per CTA; slices
 * whose ends are not 16-byte aligned go value by value); the own slice is not touched (keep it in
 * place or copy it yourself).  Order it with spl_peer_barrier like spl_spmv_peer. */
int spl_peer_pull(spl_ctx *ctx, int dtype, int world, int rank, const uint64_t *starts,
                  const void *const *slices, void *x_full_dev);
/* Row-sharded y_local = A_local * x with x left where it lives: x_slices[g] is rank
 * g's slice of x (columns [col_starts[g], col_starts[g+1]), own slice included), mapped
 * with spl_peer_open.  One kernel: every gather goes to the slice that owns the column,
 * local HBM or a peer's over NVLink; no staging copy, no collective (the sharded form
 * of `&A * &X`, src/csr/ops/mul.rs:5-60).  A_local is CSR with global column indices. */
int spl_spmv_peer(spl_ctx *ctx, const spl_mat *a_local, int world, int rank,
                  const uint64_t *col_starts, const void *const *x_slices, void *y_dev);

/* Row-sharded y_local = A_local * x for GENERAL shards (random / unstructured columns; the sharded
 * form of `&A * &X`, src/csr/ops/mul.rs:5-60), the all-gather of x fused into the product: ONE
 * persistent kernel in which one copy warp per CTA pulls the peers' slices of x over NVLink
 * (x_slices as in spl_spmv_peer) into x_full_dev with TMA bulk copies, in ring order (rank+1,
 * rank+2, ...), while the compute warps multiply the shard block by block in the same order —
 * block 0 (columns of the own slice) at once, block b as soon as its slices have landed — and
 * write y once.  The shard is passed blocked by column owner in that ring order: block b holds the
 * columns owned by the ring offsets [block_first[b], block_first[b+1]) (host array of nblocks+1
 * values, 0, 1, ..., world: block 0 is the own slice alone; NULL = one block per rank, nblocks
 * ignored); block_ptr_dev holds one row-pointer array of nrows_local+1 entries per block, block b's
 * at block_ptr_dev + b * block_ptr_stride (a multiple of 4 above nrows_local; absolute positions
 * into block_ind_dev / block_val_dev, global column indices).  The matrix reaches the compute warps
 * as TMA bulk copies of whole tiles (128 to 1024 consecutive rows of one block, more rows the
 * shorter they are), so the three arrays are 16-byte aligned, block_ind_dev / block_val_dev are
 * allocated 4 entries beyond the last stored one, and tile_entries_max[0..4] (host) bound the
 * entries any 64 / 128 / 256 / 512 / 1024 consecutive rows starting at a multiple of 32 hold in one
 * block (a tile must fit a shared-memory stage: SPL_ERR_UNSUPPORTED otherwise).  ready_dev:
 * uint32[SPL_MAX_PEERS], zeroed by the caller before epoch 1; epoch = 1, 2, 3, ... per call on this
 * buffer; nnz_local = stored entries of the shard (picks the lanes per row).  The barrier that
 * orders the peers' writes of x before the pulls is part of the kernel when flag_ptrs is given
 * (flag blocks / barrier_epoch / timeout_ms exactly as spl_peer_barrier takes them); with
 * flag_ptrs NULL run spl_peer_barrier first.  x_full_dev (ncols values) is scratch: afterwards it
 * holds the peers' slices (not the own one).  timeline_dev: NULL, or 2 + 3*nblocks zeroed uint64
 * that receive %globaltimer stamps (first copy warp past the barrier; per block: wait begins, slices
 * landed, block done on the first warp of the first CTA; the last CTA to finish) — the evidence in
 * bench.py's `sharded_spmv_gather_fused`.  The launch shape follows from the shard and the device: it is the
 * same from epoch to epoch on one ready_dev (zero it and restart at epoch 1 if anything changes). */
int spl_spmv_gather_fused(spl_ctx *ctx, int dtype, uint64_t nrows_local, int world, int rank,
                          const uint64_t *col_starts, const void *const *x_slices, int nblocks,
                          const uint32_t *block_first, const uint32_t *block_ptr_dev, uint64_t block_ptr_stride,
                          const uint32_t *tile_entries_max, const uint32_t *block_ind_dev, const void *block_val_dev, void *x_full_dev, void *y_dev,
                          uint32_t *ready_dev, uint32_t epoch, uint64_t nnz_local, void *const *flag_ptrs,
                          uint32_t barrier_epoch, uint32_t timeout_ms, uint64_t *timeline_dev);

/* The reference-facing `&A * &x` on one rank of a row-sharded matrix, with HOST vectors:
 * x_host_local is this rank's slice of x (col_starts[rank+1] - col_starts[rank] values),
 * y_host_local receives its rows of y.  The slice is uploaded into x_slices[rank] (this rank's
 * peer-visible buffer: pass the set of buffers being written, e.g. the unpublished half of a
 * double-buffered vector), the device barrier (flag_ptrs / epoch / timeout_ms as in
 * spl_peer_barrier) publishes it, and the product runs in row chunks on the compute stream while
 * finished chunks of y travel back on a second stream.  Synchronises; a timed-out barrier is
 * reported here (SPL_ERR_CUDA) and y holds NaN.  Pinned host vectors make the copies overlap. */
int spl_spmv_peer_host(spl_ctx *ctx, const spl_mat *a_local, int world, int rank, const uint64_t *col_starts,
                       void *const *x_slices, void *const *flag_ptrs, uint32_t epoch, uint32_t timeout_ms,
                       const void *x_host_local, void *y_host_local);

#ifdef __cplusplus
}
#endif
#endif /* SPL_H */
