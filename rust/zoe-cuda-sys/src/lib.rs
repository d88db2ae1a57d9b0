//! Raw bindings of `include/zoe_cuda.h` (one `extern "C"` item per declared symbol).
#![allow(non_camel_case_types)]
use core::ffi::{c_char, c_int, c_void};

#[repr(C)]
pub struct zoe_cuda_ctx {
    _private: [u8; 0],
}

pub const ZOE_CUDA_SOME: u8 = 0;
pub const ZOE_CUDA_OVERFLOWED: u8 = 1;
pub const ZOE_CUDA_UNMAPPED: u8 = 2;

pub const ZOE_CUDA_E_EMPTY_SEQUENCE: c_int = -1;
pub const ZOE_CUDA_E_GAP_OPEN_RANGE: c_int = -2;
pub const ZOE_CUDA_E_GAP_EXTEND_RANGE: c_int = -3;
pub const ZOE_CUDA_E_BAD_GAP_WEIGHTS: c_int = -4;
pub const ZOE_CUDA_E_BAD_ARG: c_int = -5;
pub const ZOE_CUDA_E_CIGAR_CAP: c_int = -6;
pub const ZOE_CUDA_E_CUDA: c_int = -7;
pub const ZOE_CUDA_E_STATE: c_int = -8;
pub const ZOE_CUDA_E_UNSUPPORTED: c_int = -9;

#[repr(C)]
#[derive(Default, Clone, Copy, Debug)]
pub struct zoe_cuda_stats {
    pub pairs: u64,
    pub cells: u64,
    pub tier8: u64,
    pub tier16: u64,
    pub tier32: u64,
    pub overflowed: u64,
    pub unmapped: u64,
    pub rerun_wide: u64,
    pub hazard: u64,
    pub window_fallback: u64,
    pub window_pinned: u64,
    pub tp_nogaps: u64,
    pub tp_banded: u64,
    pub tp_scalar: u64,
    pub tp_band_attempts: u64,
}

unsafe extern "C" {
    pub fn zoe_cuda_create(ctx: *mut *mut zoe_cuda_ctx, device_ids: *const c_int, n_devices: c_int) -> c_int;
    pub fn zoe_cuda_destroy(ctx: *mut zoe_cuda_ctx);
    pub fn zoe_cuda_last_error(ctx: *const zoe_cuda_ctx) -> *const c_char;
    pub fn zoe_cuda_set_scoring(
        ctx: *mut zoe_cuda_ctx, weights: *const i8, s: c_int, byte_to_index: *const u8, gap_open: i8, gap_extend: i8,
        profiled_is_query: c_int,
    ) -> c_int;
    pub fn zoe_cuda_set_lanes(ctx: *mut zoe_cuda_ctx, lanes_i8: c_int, lanes_i16: c_int, lanes_i32: c_int) -> c_int;
    pub fn zoe_cuda_set_width_policy(ctx: *mut zoe_cuda_ctx, first_bits: c_int, last_bits: c_int, is_unsigned: c_int) -> c_int;
    pub fn zoe_cuda_set_align_options(ctx: *mut zoe_cuda_ctx, mode: c_int, checkpoint_log2: c_int, slack: c_int) -> c_int;
    pub fn zoe_cuda_set_memory_budget(ctx: *mut zoe_cuda_ctx, scratch_bytes: u64) -> c_int;
    pub fn zoe_cuda_sneaky_snake_batch(
        ctx: *mut zoe_cuda_ctx, refs: *const u8, ref_offsets: *const u64, queries: *const u8, query_offsets: *const u64,
        n: u64, threshold: f32, out: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_set_profiled(ctx: *mut zoe_cuda_ctx, concat: *const u8, offsets: *const u64, n: u32) -> c_int;
    pub fn zoe_cuda_sw_score_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, score: *mut u32,
        status: *mut u8, tier: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_sw_align_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, score: *mut u32,
        status: *mut u8, tier: *mut u8, ref_start: *mut u32, ref_end: *mut u32, query_start: *mut u32,
        query_end: *mut u32, cigar: *mut u32, cigar_off: *mut u64, cigar_cap: u64, hazard: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_sw_score_ranges_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, score: *mut u32,
        status: *mut u8, tier: *mut u8, ref_start: *mut u32, ref_end: *mut u32, query_start: *mut u32,
        query_end: *mut u32,
    ) -> c_int;
    pub fn zoe_cuda_sw_align_3pass_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, score: *mut u32,
        status: *mut u8, tier: *mut u8, ref_start: *mut u32, ref_end: *mut u32, query_start: *mut u32,
        query_end: *mut u32, cigar: *mut u32, cigar_off: *mut u64, cigar_cap: u64,
    ) -> c_int;
    pub fn zoe_cuda_sw_score_both_strands_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, score: *mut u32,
        status: *mut u8, tier: *mut u8, strand: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_sw_score_ranges_both_strands_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, score: *mut u32,
        status: *mut u8, tier: *mut u8, ref_start: *mut u32, ref_end: *mut u32, query_start: *mut u32,
        query_end: *mut u32, strand: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_sw_align_both_strands_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, score: *mut u32,
        status: *mut u8, tier: *mut u8, ref_start: *mut u32, ref_end: *mut u32, query_start: *mut u32,
        query_end: *mut u32, cigar: *mut u32, cigar_off: *mut u64, cigar_cap: u64, hazard: *mut u8, strand: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_sw_align_3pass_both_strands_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, score: *mut u32,
        status: *mut u8, tier: *mut u8, ref_start: *mut u32, ref_end: *mut u32, query_start: *mut u32,
        query_end: *mut u32, cigar: *mut u32, cigar_off: *mut u64, cigar_cap: u64, strand: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_sw_score_best_hit_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, both_strands: c_int,
        hit: *mut u32, strand: *mut u8, score: *mut u32, status: *mut u8, tier: *mut u8, runner_up: *mut u32,
    ) -> c_int;
    pub fn zoe_cuda_sw_align_best_hit_batch(
        ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64, both_strands: c_int,
        three_pass: c_int, hit: *mut u32, strand: *mut u8, score: *mut u32, status: *mut u8, tier: *mut u8,
        runner_up: *mut u32, ref_start: *mut u32, ref_end: *mut u32, query_start: *mut u32, query_end: *mut u32,
        cigar: *mut u32, cigar_off: *mut u64, cigar_cap: u64, hazard: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_sw_score_paired_best_hit_batch(
        ctx: *mut zoe_cuda_ctx, mate1_concat: *const u8, mate1_offsets: *const u64, mate2_concat: *const u8,
        mate2_offsets: *const u64, n_pairs: u64, hit: *mut u32, strand: *mut u8, score: *mut u32, status: *mut u8,
        tier: *mut u8, runner_up: *mut u32,
    ) -> c_int;
    pub fn zoe_cuda_sw_align_paired_best_hit_batch(
        ctx: *mut zoe_cuda_ctx, mate1_concat: *const u8, mate1_offsets: *const u64, mate2_concat: *const u8,
        mate2_offsets: *const u64, n_pairs: u64, three_pass: c_int, min_insert: u32, max_insert: u32, hit: *mut u32,
        proper: *mut u8, tlen: *mut c_int, strand: *mut u8, score: *mut u32, status: *mut u8, tier: *mut u8,
        runner_up: *mut u32, ref_start: *mut u32, ref_end: *mut u32, query_start: *mut u32, query_end: *mut u32,
        cigar: *mut u32, cigar_off: *mut u64, cigar_cap: u64, hazard: *mut u8,
    ) -> c_int;
    pub fn zoe_cuda_run_ranges_staged(ctx: *mut zoe_cuda_ctx) -> c_int;
    pub fn zoe_cuda_run_3pass_staged(ctx: *mut zoe_cuda_ctx) -> c_int;
    pub fn zoe_cuda_stage_streamed(ctx: *mut zoe_cuda_ctx, streamed_concat: *const u8, offsets: *const u64, n: u64) -> c_int;
    pub fn zoe_cuda_run_score_staged(ctx: *mut zoe_cuda_ctx) -> c_int;
    pub fn zoe_cuda_run_align_staged(ctx: *mut zoe_cuda_ctx) -> c_int;
    pub fn zoe_cuda_fetch_scores(ctx: *mut zoe_cuda_ctx, score: *mut u32, status: *mut u8, tier: *mut u8) -> c_int;
    pub fn zoe_cuda_last_timing(ctx: *const zoe_cuda_ctx, total_ms: *mut f32, dp_kernel_ms: *mut f32, kernel_launches: *mut u32) -> c_int;
    pub fn zoe_cuda_last_stats(ctx: *const zoe_cuda_ctx, out: *mut zoe_cuda_stats) -> c_int;
    pub fn zoe_cuda_dpx_peak(ctx: *mut zoe_cuda_ctx, kind: c_int, giga_lane_instr_per_s: *mut f64, ms: *mut f32) -> c_int;
    pub fn zoe_cuda_stream(ctx: *mut zoe_cuda_ctx, dev_index: c_int) -> *mut c_void;
}
