//! vega_b200_sys.rs — `extern "C"` declarations of libvega_b200.so for vega (Rust).
//!
//! SOURCE ONLY: this image has no rustc/cargo (and vega needs nightly-2020-05-31 + capnpc), so
//! this file has never been compiled.  It is the binding a vega maintainer would add as
//! `src/gpu/sys.rs`; see INTEGRATION.md for the four call-site patches that use it.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

#[repr(C)] pub struct vb_ctx { _p: [u8; 0] }
#[repr(C)] pub struct vb_shuf { _p: [u8; 0] }

pub const VB_OK: i32 = 0;
pub const VB_U64: i32 = 0; pub const VB_I64: i32 = 1; pub const VB_F64: i32 = 2;
pub const VB_AGG_GROUP: i32 = 0; pub const VB_AGG_SUM: i32 = 1; pub const VB_AGG_MIN: i32 = 2;
pub const VB_AGG_MAX: i32 = 3; pub const VB_AGG_COUNT: i32 = 4; pub const VB_AGG_COGROUP: i32 = 5;
pub const VB_PART_HASH_METRO64: i32 = 0;
pub const VB_HOST: i32 = 0;
pub const VB_JOIN_LEFT_OUTER: i32 = 1; pub const VB_JOIN_RIGHT_OUTER: i32 = 2; pub const VB_JOIN_FULL_OUTER: i32 = 3;
pub const VB_JOIN_HAS_V: u8 = 1; pub const VB_JOIN_HAS_W: u8 = 2;

#[link(name = "vega_b200")]
extern "C" {
    pub fn vb_ctx_create(device_id: i32, out: *mut *mut vb_ctx) -> i32;
    pub fn vb_ctx_destroy(ctx: *mut vb_ctx) -> i32;
    pub fn vb_shuffle_create(ctx: *mut vb_ctx, shuffle_id: u64, n_map: u32, n_reduce: u32, key_dtype: i32,
                             val_dtype: i32, agg: i32, part: i32, out: *mut *mut vb_shuf) -> i32;
    pub fn vb_shuffle_set_key_width(s: *mut vb_shuf, bytes: u32) -> i32;
    pub fn vb_shuffle_map_aos(s: *mut vb_shuf, map_id: u32, rows: *const c_void, n_rows: u64, src_loc: i32) -> i32;
    pub fn vb_shuffle_map_soa(s: *mut vb_shuf, map_id: u32, keys: *const c_void, vals: *const c_void,
                              n_rows: u64, src_loc: i32) -> i32;
    pub fn vb_shuffle_seal(s: *mut vb_shuf) -> i32;
    pub fn vb_shuffle_reduce_size(s: *mut vb_shuf, reduce_id: u32, n_keys: *mut u64, n_vals: *mut u64) -> i32;
    pub fn vb_shuffle_reduce(s: *mut vb_shuf, reduce_id: u32, out_keys: *mut c_void, out_combined: *mut c_void,
                             out_offsets: *mut u64, out_vals: *mut c_void, dst_loc: i32) -> i32;
    pub fn vb_join_size(left: *mut vb_shuf, right: *mut vb_shuf, reduce_id: u32, n_out: *mut u64) -> i32;
    pub fn vb_join(left: *mut vb_shuf, right: *mut vb_shuf, reduce_id: u32, out_k: *mut c_void, out_v: *mut c_void,
                   out_w: *mut c_void, dst_loc: i32) -> i32;
    // CoGroupedRdd::compute (PairRdd::cogroup) and Spark's outer joins, one reduce partition
    pub fn vb_cogroup_size(left: *mut vb_shuf, right: *mut vb_shuf, reduce_id: u32, n_keys: *mut u64,
                           n_left_vals: *mut u64, n_right_vals: *mut u64) -> i32;
    pub fn vb_cogroup(left: *mut vb_shuf, right: *mut vb_shuf, reduce_id: u32, out_keys: *mut c_void, out_offs_l: *mut u64,
                      out_vals_l: *mut c_void, out_offs_r: *mut u64, out_vals_r: *mut c_void, dst_loc: i32) -> i32;
    pub fn vb_join_outer_size(left: *mut vb_shuf, right: *mut vb_shuf, reduce_id: u32, kind: i32, n_out: *mut u64) -> i32;
    pub fn vb_join_outer(left: *mut vb_shuf, right: *mut vb_shuf, reduce_id: u32, kind: i32, out_k: *mut c_void,
                         out_v: *mut c_void, out_w: *mut c_void, out_valid: *mut u8 /* may be null */, dst_loc: i32) -> i32;
    // N1: bincode blobs (the payload format of SHUFFLE_CACHE)
    pub fn vb_shuffle_reduce_blob_size(s: *mut vb_shuf, reduce_id: u32, n_bytes: *mut u64) -> i32;
    pub fn vb_shuffle_reduce_blob(s: *mut vb_shuf, reduce_id: u32, out_blob: *mut c_void, dst_loc: i32) -> i32;
    pub fn vb_shuffle_map_blob(s: *mut vb_shuf, map_id: u32, blob: *const c_void, n_bytes: u64, src_loc: i32) -> i32;
    // one process per GPU: pack + all-to-all-v, or the fused exchange over peer memory
    pub fn vb_shuffle_set_dist(s: *mut vb_shuf, rank: u32, world: u32) -> i32;
    pub fn vb_shuffle_export_prepare(s: *mut vb_shuf, counts: *mut u64) -> i32;
    pub fn vb_shuffle_export_buffers(s: *mut vb_shuf, keys_dev: *mut *mut c_void, vals_dev: *mut *mut c_void) -> i32;
    pub fn vb_shuffle_import(s: *mut vb_shuf, keys_dev: *const c_void, vals_dev: *const c_void, counts: *const u64) -> i32;
    pub fn vb_ctx_arena_reserve(ctx: *mut vb_ctx, bytes: u64, handle_out: *mut c_void, generation: *mut u64) -> i32;
    pub fn vb_ctx_peer_open(ctx: *mut vb_ctx, peer_rank: u32, handle: *const c_void, generation: u64, is_self: i32) -> i32;
    pub fn vb_shuffle_export_counts(s: *mut vb_shuf, counts: *mut u64) -> i32;
    pub fn vb_shuffle_export_direct(s: *mut vb_shuf, dst_row_offset: *const u64, dst_total_rows: *const u64) -> i32;
    pub fn vb_shuffle_import_arena(s: *mut vb_shuf, counts: *const u64) -> i32;
    // the exchange inside the library: NCCL communicator per context (unique id handed out by vega's tracker channel)
    pub fn vb_comm_unique_id(id_out: *mut c_void /* 128 bytes */) -> i32;
    pub fn vb_ctx_comm_init(ctx: *mut vb_ctx, unique_id: *const c_void, rank: u32, world: u32) -> i32;
    pub fn vb_ctx_comm_destroy(ctx: *mut vb_ctx) -> i32;
    pub fn vb_shuffle_exchange(s: *mut vb_shuf, mode: i32 /* VB_XCHG_AUTO = 0 */) -> i32;
    pub fn vb_ctx_arena_release_retired(ctx: *mut vb_ctx) -> i32;
    pub fn vb_ctx_trim(ctx: *mut vb_ctx, keep_bytes: u64) -> i32;
    // device-resident source (Context::range)
    pub fn vb_range_len(start: u64, end: u64, step: u64) -> u64;
    pub fn vb_range(ctx: *mut vb_ctx, out_dev: *mut c_void, start: u64, end: u64, step: u64) -> i32;
    pub fn vb_shuffle_free(s: *mut vb_shuf) -> i32;
    pub fn vb_last_error() -> *const c_char;
    pub fn vb_get_partition(key: u64, key_width: u32, n_reduce: u32) -> u32;
}
