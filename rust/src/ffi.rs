//! The `extern "C"` block: one to one with `include/spl.h` (the same text as INTEGRATION.md section 2).
#![allow(non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct spl_ctx { _p: [u8; 0] }
#[repr(C)] pub struct spl_mat { _p: [u8; 0] }
#[repr(C)] pub struct spl_coo { _p: [u8; 0] }

pub const SPL_OK: c_int = 0;
pub const SPL_CSR: c_int = 0; pub const SPL_CSC: c_int = 1;
pub const SPL_F32: c_int = 0; pub const SPL_F64: c_int = 1;
pub const SPL_SPMV_AUTO: c_int = 0; pub const SPL_SPMV_VECTOR: c_int = 1; pub const SPL_SPMV_MERGE: c_int = 2;
pub const SPL_SPMV_SPLIT: c_int = 3; pub const SPL_SPMV_SLICED: c_int = 4;   // spl_spmv_ex: kernel | lanes << 8
pub const SPL_SPMV_STREAM: c_int = 5; pub const SPL_SPMV_SCATTER: c_int = 6;

extern "C" {
    pub fn spl_ctx_create(device: c_int, stream: *mut c_void, out: *mut *mut spl_ctx) -> c_int;
    pub fn spl_ctx_destroy(ctx: *mut spl_ctx) -> c_int;
    pub fn spl_ctx_sync(ctx: *mut spl_ctx) -> c_int;
    pub fn spl_ctx_trim(ctx: *mut spl_ctx) -> c_int;
    pub fn spl_host_alloc(bytes: u64, out: *mut *mut c_void) -> c_int;
    pub fn spl_host_free(p: *mut c_void) -> c_int;
    pub fn spl_host_register(p: *mut c_void, bytes: u64) -> c_int;
    pub fn spl_host_unregister(p: *mut c_void) -> c_int;
    pub fn spl_last_error(ctx: *const spl_ctx) -> *const c_char;
    pub fn spl_invalid_reason(ctx: *const spl_ctx) -> c_int;
    pub fn spl_launch_count(ctx: *const spl_ctx) -> u64;
    pub fn spl_mat_from_coo(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nrows: u64, ncols: u64,
        len: u64, row: *const u64, col: *const u64, val: *const c_void,
        dedup: c_int, dropzero: c_int, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_from_coo_dev(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nrows: u64, ncols: u64,
        len: u64, row: *const u32, col: *const u32, val: *const c_void,
        dedup: c_int, dropzero: c_int, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_from_compressed(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nrows: u64, ncols: u64,
        ptr_len: u64, ptr: *const u64, ind_len: u64, ind: *const u64,
        val_len: u64, val: *const c_void, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_from_compressed_dev(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nrows: u64,
        ncols: u64, nnz: u64, ptr: *const u32, ind: *const u32, val: *const c_void,
        validate: c_int, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_from_compressed_dev64(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nrows: u64,
        ncols: u64, nnz: u64, ptr: *const u64, ind: *const u32, val: *const c_void,
        validate: c_int, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_device_ptr64(m: *const spl_mat, ptr64: *mut *const u64) -> c_int;
    pub fn spl_mat_eye(ctx: *mut spl_ctx, format: c_int, dtype: c_int, size: u64, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_convert(ctx: *mut spl_ctx, m: *const spl_mat, format: c_int, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_transpose(ctx: *mut spl_ctx, m: *const spl_mat, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_add(ctx: *mut spl_ctx, a: *const spl_mat, b: *const spl_mat, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_sub(ctx: *mut spl_ctx, a: *const spl_mat, b: *const spl_mat, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_mul(ctx: *mut spl_ctx, a: *const spl_mat, b: *const spl_mat, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_mat_neg(ctx: *mut spl_ctx, a: *const spl_mat, out: *mut *mut spl_mat) -> c_int;
    pub fn spl_spmv(ctx: *mut spl_ctx, a: *const spl_mat, x_dev: *const c_void, y_dev: *mut c_void) -> c_int;
    pub fn spl_spmv_ex(ctx: *mut spl_ctx, a: *const spl_mat, x_dev: *const c_void, y_dev: *mut c_void, kernel: c_int) -> c_int;
    pub fn spl_spmv_host(ctx: *mut spl_ctx, a: *const spl_mat, x: *const c_void, y: *mut c_void) -> c_int;
    pub fn spl_spmv_choice(ctx: *mut spl_ctx, a: *const spl_mat, kernel: *mut c_int, lanes: *mut c_int) -> c_int;
    pub fn spl_mat_info(m: *const spl_mat, format: *mut c_int, dtype: *mut c_int,
        nrows: *mut u64, ncols: *mut u64, nnz: *mut u64) -> c_int;
    pub fn spl_mat_download(ctx: *mut spl_ctx, m: *const spl_mat, ptr: *mut u64, ind: *mut u64, val: *mut c_void) -> c_int;
    pub fn spl_mat_set_values(ctx: *mut spl_ctx, m: *mut spl_mat, val: *const c_void) -> c_int;
    pub fn spl_mat_device_ptrs(m: *const spl_mat, ptr: *mut *const u32, ind: *mut *const u32, val: *mut *const c_void) -> c_int;
    pub fn spl_mat_to_coo(ctx: *mut spl_ctx, m: *const spl_mat, row: *mut u64, col: *mut u64, val: *mut c_void) -> c_int;
    pub fn spl_mat_to_coo_dev(ctx: *mut spl_ctx, m: *const spl_mat, row: *mut u32, col: *mut u32, val: *mut c_void) -> c_int;
    pub fn spl_mat_read_entries(ctx: *mut spl_ctx, m: *const spl_mat, start: u64, count: u64,
        row: *mut u64, col: *mut u64, val: *mut c_void) -> c_int;
    pub fn spl_mat_free(ctx: *mut spl_ctx, m: *mut spl_mat) -> c_int;
    // CooMatrix storage streamed to the device while it is filled (SURVEY.md 8f-4), section 4
    pub fn spl_coo_create(ctx: *mut spl_ctx, dtype: c_int, nrows: u64, ncols: u64, capacity: u64,
        out: *mut *mut spl_coo) -> c_int;
    pub fn spl_coo_free(coo: *mut spl_coo) -> c_int;
    pub fn spl_coo_last_error(coo: *const spl_coo) -> *const c_char;
    pub fn spl_coo_push(coo: *mut spl_coo, row: u64, col: u64, value: *const c_void) -> c_int;
    pub fn spl_coo_extend(coo: *mut spl_coo, len: u64, row: *const u64, col: *const u64, val: *const c_void) -> c_int;
    pub fn spl_coo_reserve(coo: *mut spl_coo, capacity: u64) -> c_int;
    pub fn spl_coo_truncate(coo: *mut spl_coo, len: u64) -> c_int;
    pub fn spl_coo_len(coo: *const spl_coo) -> u64;
    pub fn spl_coo_capacity(coo: *const spl_coo) -> u64;
    pub fn spl_coo_streamed(coo: *const spl_coo) -> u64;
    pub fn spl_coo_invalidate(coo: *mut spl_coo, first: u64) -> c_int;
    pub fn spl_coo_host_ptrs(coo: *const spl_coo, row: *mut *const u64, col: *mut *const u64,
        val: *mut *const c_void) -> c_int;
    pub fn spl_mat_from_coo_builder(ctx: *mut spl_ctx, coo: *mut spl_coo, format: c_int, dedup: c_int,
        dropzero: c_int, out: *mut *mut spl_mat) -> c_int;
    // row sharding across the GPUs of one box (one process per GPU), section 7
    pub fn spl_coo_route_dev(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nrows: u64, ncols: u64,
        len: u64, row: *const u32, col: *const u32, val: *const c_void, world: c_int,
        major_starts: *const u64, keys_out: *mut u64, vals_out: *mut c_void, counts: *mut u64) -> c_int;
    pub fn spl_coo_route_count_dev(ctx: *mut spl_ctx, format: c_int, nrows: u64, ncols: u64, len: u64,
        row: *const u32, col: *const u32, world: c_int, major_starts: *const u64, counts: *mut u64) -> c_int;
    pub fn spl_coo_route_peers_dev(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nrows: u64, ncols: u64,
        len: u64, row: *const u32, col: *const u32, val: *const c_void, world: c_int,
        major_starts: *const u64, key_bufs: *const *mut c_void, val_bufs: *const *mut c_void,
        dst_offsets: *const u64) -> c_int;
    pub fn spl_mat_from_packed_dev(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nrows: u64, ncols: u64,
        len: u64, keys: *const u64, vals: *const c_void, dedup: c_int, dropzero: c_int,
        out: *mut *mut spl_mat) -> c_int;
    pub fn spl_peer_alloc(ctx: *mut spl_ctx, bytes: u64, dev_ptr: *mut *mut c_void, handle: *mut u8) -> c_int;
    pub fn spl_peer_open(ctx: *mut spl_ctx, handle: *const u8, peer_ptr: *mut *mut c_void) -> c_int;
    pub fn spl_peer_close(ctx: *mut spl_ctx, peer_ptr: *mut c_void) -> c_int;
    pub fn spl_peer_free(ctx: *mut spl_ctx, dev_ptr: *mut c_void) -> c_int;
    pub fn spl_peer_barrier(ctx: *mut spl_ctx, world: c_int, rank: c_int, flag_ptrs: *const *mut c_void,
        epoch: u32, timeout_ms: u32) -> c_int;
    pub fn spl_peer_barrier_status(ctx: *mut spl_ctx, timed_out: *mut c_int) -> c_int;
    pub fn spl_peer_pull(ctx: *mut spl_ctx, dtype: c_int, world: c_int, rank: c_int, starts: *const u64,
        slices: *const *const c_void, x_full_dev: *mut c_void) -> c_int;
    pub fn spl_peer_gather_rows(ctx: *mut spl_ctx, format: c_int, dtype: c_int, nmajor: u64, nminor: u64, world: c_int,
        rank: c_int, starts: *const u64, shard_nnz: *const u64, ptr_slices: *const *const c_void,
        ind_slices: *const *const c_void, val_slices: *const *const c_void, by: *const spl_mat,
        out: *mut *mut spl_mat) -> c_int;
    pub fn spl_spmv_peer(ctx: *mut spl_ctx, a_local: *const spl_mat, world: c_int, rank: c_int,
        col_starts: *const u64, x_slices: *const *const c_void, y_dev: *mut c_void) -> c_int;
    pub fn spl_peer_barrier_halo(ctx: *mut spl_ctx, world: c_int, rank: c_int, flag_ptrs: *const *mut c_void,
        epoch: u32, timeout_ms: u32, dtype: c_int, starts: *const u64, x_slices: *const *mut c_void,
        halo_left: u64, halo_right: u64) -> c_int;
    pub fn spl_spmv_window(ctx: *mut spl_ctx, a: *const spl_mat, x_window_dev: *const c_void, window_start: u64,
        window_len: u64, y_dev: *mut c_void) -> c_int;
    pub fn spl_spmv_footprint(ctx: *mut spl_ctx, a: *const spl_mat, col_min: *mut u64, col_max: *mut u64) -> c_int;
    pub fn spl_spmv_transpose_window(ctx: *mut spl_ctx, a: *const spl_mat, x_dev: *const c_void,
        y_window_dev: *mut c_void) -> c_int;
    pub fn spl_peer_reduce_windows(ctx: *mut spl_ctx, dtype: c_int, world: c_int, rank: c_int, col_starts: *const u64,
        windows: *const u64, partials: *const *const c_void, flag_ptrs: *const *mut c_void, epoch: u32,
        timeout_ms: u32, y_local_dev: *mut c_void) -> c_int;
    pub fn spl_spmv_gather_fused(ctx: *mut spl_ctx, dtype: c_int, nrows_local: u64, world: c_int, rank: c_int,
        col_starts: *const u64, x_slices: *const *const c_void, nblocks: c_int, block_first: *const u32,
        block_ptr: *const u32, block_ptr_stride: u64, tile_entries_max: *const u32, block_ind: *const u32,
        block_val: *const c_void, x_full_dev: *mut c_void, y_dev: *mut c_void, ready_dev: *mut u32, epoch: u32,
        nnz_local: u64, flag_ptrs: *const *mut c_void, barrier_epoch: u32, timeout_ms: u32,
        timeline_dev: *mut u64) -> c_int;
    pub fn spl_spmv_peer_host(ctx: *mut spl_ctx, a_local: *const spl_mat, world: c_int, rank: c_int,
        col_starts: *const u64, x_slices: *const *mut c_void, flag_ptrs: *const *mut c_void, epoch: u32,
        timeout_ms: u32, x_host_local: *const c_void, y_host_local: *mut c_void) -> c_int;
}
