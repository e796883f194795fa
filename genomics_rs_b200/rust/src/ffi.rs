//! ffi.rs -- NOT COMPILED IN THIS ENVIRONMENT.  `extern "C"` declarations of include/gxalign.h.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int};

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct gx_scores {
    pub s_match: i32,
    pub s_mismatch: i32,
    pub g: i32,
    pub h: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct gx_result {
    pub score: i64,
    pub start_i: u64,
    pub start_j: u64,
    pub end_i: u64,
    pub end_j: u64,
    pub n_ops: u64,
    pub matches: u64,
    pub mismatches: u64,
    pub gap_extensions: u64,
    pub opening_gaps: u64,
    pub lcs_at_first_max: u64,
    pub fill_ms: f64,
    pub walk_ms: f64,
}

pub const GX_OK: c_int = 0;
pub const GX_FLAG_TRACEBACK: c_int = 1;
pub const GX_FLAG_LCS_AT_MAX: c_int = 2; // gx_result.lcs_at_first_max = alignment_table's 2nd return value
pub const GX_BAND_HANDLE_BYTES: usize = 64;

/// opaque: this process's column bands of one wide global table (include/gxalign.h, gx_band_*)
#[repr(C)]
pub struct gx_band {
    _private: [u8; 0],
}

extern "C" {
    pub fn gx_init(device: c_int) -> c_int;
    pub fn gx_shutdown();
    pub fn gx_strerror(status: c_int) -> *const c_char;
    pub fn gx_last_error() -> *const c_char;
    pub fn gx_align_pair(
        s1: *const u8, m: u64, s2: *const u8, n: u64, sc: gx_scores, is_local: c_int, flags: c_int,
        out: *mut gx_result, ops: *mut u8, ops_cap: u64,
    ) -> c_int;
    pub fn gx_align_batch(
        seq_blob: *const u8, blob_len: u64, off1: *const u64, len1: *const u64, off2: *const u64, len2: *const u64,
        n_pairs: u64, sc: gx_scores, is_local: c_int, flags: c_int, out: *mut gx_result, ops_blob: *mut u8,
        ops_off: *const u64,
    ) -> c_int;
    // one very long pair, global, score only, column-banded over the GPUs of a node (one process per GPU)
    pub fn gx_band_range(n_total: u64, n_bands: c_int, band: c_int, col0: *mut u64, width: *mut u64) -> c_int;
    pub fn gx_band_create(m: u64, n_total: u64, n_bands: c_int, first_band: c_int, last_band: c_int, sc: gx_scores,
                          band: *mut *mut gx_band) -> c_int;
    pub fn gx_band_export(band: *mut gx_band, handle: *mut u8, handle_cap: u64) -> c_int;
    pub fn gx_band_connect(band: *mut gx_band, left_handle: *const u8, right_handle: *const u8) -> c_int;
    pub fn gx_band_upload(band: *mut gx_band, s1: *const u8, s2: *const u8) -> c_int;
    pub fn gx_band_execute(band: *mut gx_band) -> c_int;
    pub fn gx_band_score(band: *mut gx_band, score: *mut i64, valid: *mut c_int) -> c_int;
    pub fn gx_band_destroy(band: *mut gx_band);
    pub fn gx_nw_score_banded(s1: *const u8, m: u64, s2: *const u8, n: u64, sc: gx_scores, n_bands: c_int,
                              score: *mut i64) -> c_int;
    pub fn gx_debug_planes(s1: *const u8, m: u64, s2: *const u8, n: u64, sc: gx_scores, is_local: c_int,
                           insert_scores: *mut i64, delete_scores: *mut i64, sub_scores: *mut i64) -> c_int;
    pub fn gx_score_batch(
        seq_blob: *const u8, blob_len: u64, off1: *const u64, len1: *const u64, off2: *const u64, len2: *const u64,
        n_pairs: u64, sc: gx_scores, is_local: c_int, scores: *mut i64,
    ) -> c_int;
    // gx_score_batch plus each pair's start cell (local: last argmax, (m, n) when the maximum is 0; global: (m, n))
    pub fn gx_score_batch_cells(
        seq_blob: *const u8, blob_len: u64, off1: *const u64, len1: *const u64, off2: *const u64, len2: *const u64,
        n_pairs: u64, sc: gx_scores, is_local: c_int, scores: *mut i64, start_i: *mut u64, start_j: *mut u64,
    ) -> c_int;
}
