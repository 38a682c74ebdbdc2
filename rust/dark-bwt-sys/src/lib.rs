//! Raw bindings to include/dark_bwt.h.  UNCOMPILED in this image (no Rust toolchain).
#![allow(non_camel_case_types)]
extern crate libc;
use libc::{c_char, c_int, c_void};

pub const DARK_BWT_OK: c_int = 0;
pub const DARK_BWT_MAX_ROUNDS: usize = 40;

#[repr(C)]
pub struct dark_bwt_ctx { _private: [u8; 0] }

#[repr(C)]
pub struct dark_bwt_stats {
    pub n: u64,
    pub sigma: u32,
    pub bits_per_symbol: u32,
    pub symbols_per_key: u32,
    pub initial_symbols: u32,
    pub pair_rounds: u32,
    pub rounds: u32,
    pub sort_passes: u32,
    pub kernel_launches: u32,
    pub active: [u64; DARK_BWT_MAX_ROUNDS],
    pub passes: [u32; DARK_BWT_MAX_ROUNDS],
    pub sorted_elements: u64,
    pub device_ms: f32,
    pub init_ms: f32,
    pub sort_ms: f32,
    pub pass_ms: f32,
    pub keybuild_ms: f32,
    pub rerank_ms: f32,
    pub emit_ms: f32,
    pub h2d_ms: f32,
    pub d2h_ms: f32,
    pub gen_passes: u32,
    pub gen_pass_ms: f32,
    pub gen_elements: u64,
    pub host_syncs: u32,
    pub reserved_: u32,
}

#[repr(C)]
pub struct dark_bwt_dc_info {
    pub init: [u64; 256],
    pub mtf_symbols: [u8; 256],
    pub num_unique: u32,
    pub reserved_: u32,
    pub num_items: u64,
    pub device_ms: f32,
    pub reserved2_: u32,
}

extern "C" {
    pub fn dark_bwt_abi_version() -> c_int;
    pub fn dark_bwt_dc_encode(ctx: *mut dark_bwt_ctx, bwt: *const u8, n: u64, dist_out: *mut u32, item_pos: *mut u32,
                              item_dist: *mut u32, item_sym: *mut u8, item_rank: *mut u8, info: *mut dark_bwt_dc_info) -> c_int;
    pub fn dark_bwt_dc_encode_device(ctx: *mut dark_bwt_ctx, d_bwt: *const u8, n: u64, d_dist_out: *mut u32, d_item_pos: *mut u32,
                                     d_item_dist: *mut u32, d_item_sym: *mut u8, d_item_rank: *mut u8, info: *mut dark_bwt_dc_info) -> c_int;
    pub fn dark_bwt_forward_dc(ctx: *mut dark_bwt_ctx, text: *const u8, n: u64, bwt_out: *mut u8, origin_out: *mut u64,
                               dist_out: *mut u32, item_pos: *mut u32, item_dist: *mut u32, item_sym: *mut u8, item_rank: *mut u8,
                               info: *mut dark_bwt_dc_info, stats: *mut dark_bwt_stats) -> c_int;
    pub fn dark_bwt_create(max_n: u64, device: c_int, out: *mut *mut dark_bwt_ctx) -> c_int;
    pub fn dark_bwt_create_ex(max_n: u64, device: c_int, flags: u32, out: *mut *mut dark_bwt_ctx) -> c_int;
    pub fn dark_bwt_capacity(ctx: *const dark_bwt_ctx) -> u64;
    pub fn dark_bwt_forward(ctx: *mut dark_bwt_ctx, text: *const u8, n: u64, bwt_out: *mut u8,
                            origin_out: *mut u64, sa_out: *mut u32, stats: *mut dark_bwt_stats) -> c_int;
    pub fn dark_bwt_forward_batch(ctx: *mut dark_bwt_ctx, texts: *const *const u8, ns: *const u64, bwt_outs: *const *mut u8,
                                  origins_out: *mut u64, sa_outs: *const *mut u32, count: u64, stats: *mut dark_bwt_stats) -> c_int;
    pub fn dark_bwt_forward_many(ctx: *mut dark_bwt_ctx, texts: *const *const u8, ns: *const u64, bwt_outs: *const *mut u8,
                                 origins_out: *mut u64, count: u64, stats: *mut dark_bwt_stats) -> c_int;
    pub fn dark_bwt_forward_many_device(ctx: *mut dark_bwt_ctx, d_text: *const u8, d_starts: *const u32, count: u64,
                                        d_bwt_out: *mut u8, d_origins_out: *mut u64, d_sa_out: *mut u32,
                                        stats: *mut dark_bwt_stats) -> c_int;
    pub fn dark_bwt_forward_device(ctx: *mut dark_bwt_ctx, d_text: *const u8, n: u64, d_bwt_out: *mut u8,
                                   origin_out: *mut u64, d_sa_out: *mut u32, stats: *mut dark_bwt_stats) -> c_int;
    pub fn dark_bwt_inverse(ctx: *mut dark_bwt_ctx, bwt: *const u8, n: u64, origin: u64, text_out: *mut u8) -> c_int;
    pub fn dark_bwt_inverse_batch(ctx: *mut dark_bwt_ctx, bwts: *const *const u8, ns: *const u64, origins: *const u64,
                                  text_outs: *const *mut u8, count: u64, ms_out: *mut f32) -> c_int;
    pub fn dark_bwt_inverse_many(ctx: *mut dark_bwt_ctx, bwts: *const *const u8, ns: *const u64, origins: *const u64,
                                 text_outs: *const *mut u8, count: u64, ms_out: *mut f32) -> c_int;
    pub fn dark_bwt_inverse_many_device(ctx: *mut dark_bwt_ctx, d_bwt: *const u8, d_starts: *const u32, d_origins: *const u64,
                                        count: u64, d_text_out: *mut u8, ms_out: *mut f32) -> c_int;
    pub fn dark_bwt_reuse(ctx: *mut dark_bwt_ctx, words_out: *mut *mut u32, count_out: *mut u64) -> c_int;
    pub fn dark_bwt_destroy(ctx: *mut dark_bwt_ctx);
    pub fn dark_bwt_strerror(code: c_int) -> *const c_char;
    pub fn dark_bwt_last_error(ctx: *const dark_bwt_ctx) -> *const c_char;
    pub fn dark_bwt_stream(ctx: *const dark_bwt_ctx) -> *mut c_void;
}
