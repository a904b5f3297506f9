//! ffi.rs -- `extern "C"` declarations mirroring include/nafgpu.h 1:1.
//!
//! UNBUILT: the build image has no cargo/rustc.  This file documents the binding a maintainer of
//! althonos/nafcodec would add as `nafcodec/src/decoder/device/ffi.rs` (feature `cuda`).
#![allow(non_camel_case_types, dead_code)]

use std::os::raw::{c_char, c_int, c_void};

pub const NAFGPU_OK: c_int = 0;
pub const NAFGPU_ERR_UNEXPECTED_EOF: c_int = -1;
pub const NAFGPU_ERR_INVALID_DATA: c_int = -2;
pub const NAFGPU_ERR_PARSE: c_int = -3;
pub const NAFGPU_ERR_UTF8: c_int = -4;
pub const NAFGPU_ERR_CUDA: c_int = -5;
pub const NAFGPU_ERR_NOMEM: c_int = -6;
pub const NAFGPU_ERR_ARGUMENT: c_int = -7;
pub const NAFGPU_ERR_NO_DEVICE: c_int = -8;
pub const NAFGPU_ERR_UNSUPPORTED: c_int = -9;

pub const NAFGPU_WANT_ID: u32 = 1;
pub const NAFGPU_WANT_COMMENT: u32 = 2;
pub const NAFGPU_WANT_SEQUENCE: u32 = 4;
pub const NAFGPU_WANT_QUALITY: u32 = 8;
pub const NAFGPU_WANT_MASK: u32 = 16;

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct nafgpu_header {
    pub format_version: i32,
    pub sequence_type: i32,
    pub flags: u32,
    pub name_separator: i32,
    pub line_length: u64,
    pub number_of_sequences: u64,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct nafgpu_section {
    pub data: *const u8,
    pub compressed_size: u64,
    pub original_size: u64,
    pub present: i32,
    pub _pad: i32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct nafgpu_archive {
    pub header: nafgpu_header,
    /// Id, Comment, Length, Mask, Sequence, Quality (decoder/mod.rs:237-242)
    pub sections: [nafgpu_section; 6],
}

#[repr(C)]
pub struct nafgpu_result {
    pub n_records: u64,
    pub n_ids: u64,
    pub n_comments: u64,
    pub n_lengths: u64,
    pub total_residues: u64,
    pub ids: *const u8,
    pub id_offsets: *const u64,
    pub comments: *const u8,
    pub comment_offsets: *const u64,
    pub lengths: *const u64,
    pub record_offsets: *const u64,
    pub sequence: *const u8,
    pub quality: *const u8,
    pub first_bad_record: u64,
    pub record_status: i32,
    pub status: i32, // 0, or why this archive of the batch could not be decoded
}

/// `nafgpu_text` (include/nafgpu.h): FASTA / FASTQ text of one archive in pinned host memory owned by the context.
#[repr(C)]
pub struct nafgpu_text {
    pub data: *const u8,
    pub size: u64,
    pub format: i32,
    pub status: i32,
    pub first_bad_record: u64,
}

pub const NAFGPU_TEXT_AUTO: c_int = 0;
pub const NAFGPU_TEXT_FASTA: c_int = 1;
pub const NAFGPU_TEXT_FASTQ: c_int = 2;
pub const NAFGPU_LINE_LENGTH_FROM_HEADER: u64 = u64::MAX;

#[repr(C)]
pub struct nafgpu_ctx {
    _private: [u8; 0],
}

/// Several contexts and their host threads behind submit / wait / release (include/nafgpu.h, "pipeline").
#[repr(C)]
pub struct nafgpu_pipeline {
    _private: [u8; 0],
}

/// Input of `nafgpu_pack`: what `Encoder::push` receives for every record, concatenated (encoder/mod.rs:265-300).
#[repr(C)]
pub struct nafgpu_pack_input {
    pub sequence: *const u8,
    pub lengths: *const u64,
    pub n_records: u64,
    pub n_residues: u64,
    pub sequence_type: i32, // 0 dna, 1 rna
    pub extract_mask: i32,
}

/// The Sequence, Length and Mask streams as the writers would hand them to zstd (encoder/writer.rs:21-90, mod.rs:37-44).
#[repr(C)]
pub struct nafgpu_pack_result {
    pub packed: *const u8,
    pub packed_size: u64,
    pub length_words: *const u8,
    pub length_size: u64,
    pub mask: *const u8,
    pub mask_size: u64,
    pub n_mask_runs: u64,
    pub first_invalid: u64,
}

/// `nafgpu_counts` (include/nafgpu.h): per-archive counters of the job that was run.
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct nafgpu_counts {
    pub n_records: u64,
    pub n_ids: u64,
    pub n_comments: u64,
    pub n_lengths: u64,
    pub total_residues: u64,
    pub id_bytes: u64,
    pub comment_bytes: u64,
    pub first_bad_record: u64,
    pub record_status: i32,
    pub status: i32,
}

pub const NAFGPU_SEC_ID: i32 = 0;
pub const NAFGPU_SEC_COMMENT: i32 = 1;
pub const NAFGPU_SEC_SEQUENCE: i32 = 4;
pub const NAFGPU_SEC_QUALITY: i32 = 5;
pub const NAFGPU_EXPORT_FLAT: i32 = 0;
pub const NAFGPU_EXPORT_ROWS: i32 = 1;
pub const NAFGPU_EXPORT_OFFSETS: i32 = 2;

/// `nafgpu_export` (include/nafgpu.h): one export of the decoded job into device memory the caller owns.
#[repr(C)]
pub struct nafgpu_export {
    pub field: i32,
    pub layout: i32,
    pub table: [u8; 256],
    pub pad: u8,
    pub _pad: [u8; 7],
    pub out: *mut c_void,         // DEVICE memory
    pub out_bytes: u64,
    pub rows: *const i64,         // DEVICE, ROWS: n_rows (record, start) pairs
    pub n_rows: u64,
    pub row_length: u64,
}

extern "C" {
    pub fn nafgpu_ctx_create(device: c_int, out: *mut *mut nafgpu_ctx) -> c_int;
    pub fn nafgpu_ctx_destroy(ctx: *mut nafgpu_ctx);
    pub fn nafgpu_last_error(ctx: *const nafgpu_ctx) -> *const c_char;
    pub fn nafgpu_strerror(status: c_int) -> *const c_char;
    pub fn nafgpu_host_alloc(bytes: usize) -> *mut c_void;
    pub fn nafgpu_host_free(p: *mut c_void);
    pub fn nafgpu_decode(
        ctx: *mut nafgpu_ctx,
        archive: *const nafgpu_archive,
        want: u32,
        out: *mut nafgpu_result,
    ) -> c_int;
    pub fn nafgpu_decode_batch(
        ctx: *mut nafgpu_ctx,
        archives: *const nafgpu_archive,
        n: u32,
        want: u32,
        out: *mut nafgpu_result,
    ) -> c_int;
    /// prepare + run + FASTA/FASTQ formatting on the device (what a `Decoder::to_fasta` helper would call)
    pub fn nafgpu_format_batch(
        ctx: *mut nafgpu_ctx,
        archives: *const nafgpu_archive,
        n: u32,
        want: u32,
        format: c_int,
        line_length: u64,
        out: *mut nafgpu_text,
    ) -> c_int;
    pub fn nafgpu_job_prepare(ctx: *mut nafgpu_ctx, archives: *const nafgpu_archive, n: u32, want: u32) -> c_int;
    pub fn nafgpu_job_run(ctx: *mut nafgpu_ctx) -> c_int;
    /// Bounded-memory fetch of records [first, first + count) of one archive of the job that was run (nafgpu.h).
    pub fn nafgpu_job_fetch_window(
        ctx: *mut nafgpu_ctx,
        archive: u32,
        first: u64,
        count: u64,
        max_bytes: u64,
        out: *mut nafgpu_result,
    ) -> c_int;
    pub fn nafgpu_pipeline_create(device: c_int, lanes: u32, out: *mut *mut nafgpu_pipeline) -> c_int;
    pub fn nafgpu_pipeline_destroy(p: *mut nafgpu_pipeline);
    /// returns a ticket (>= 0) or a negative status; the archives are borrowed until `wait` returns
    pub fn nafgpu_pipeline_submit(p: *mut nafgpu_pipeline, archives: *const nafgpu_archive, n: u32, want: u32) -> i64;
    pub fn nafgpu_pipeline_wait(p: *mut nafgpu_pipeline, ticket: i64, out: *mut nafgpu_result, n: u32) -> c_int;
    pub fn nafgpu_pipeline_release(p: *mut nafgpu_pipeline, ticket: i64) -> c_int;
    pub fn nafgpu_pipeline_last_error(p: *const nafgpu_pipeline) -> *const c_char;
    pub fn nafgpu_pipeline_lanes(p: *const nafgpu_pipeline) -> u32;
    pub fn nafgpu_pack(ctx: *mut nafgpu_ctx, input: *const nafgpu_pack_input, out: *mut nafgpu_pack_result) -> c_int;
    pub fn nafgpu_job_counts(ctx: *mut nafgpu_ctx, out: *mut nafgpu_counts, n: u32) -> c_int;
    /// enqueued on `stream` (a cudaStream_t; null = the context's stream), ordered after the run and before the context's next call
    pub fn nafgpu_job_export(ctx: *mut nafgpu_ctx, spec: *const nafgpu_export, stream: *mut c_void) -> c_int;
    /// a device ticket: the lane decodes and reads the counters, the sub-batch stays in its arena until release
    pub fn nafgpu_pipeline_submit_device(p: *mut nafgpu_pipeline, archives: *const nafgpu_archive, n: u32, want: u32) -> i64;
    /// the archives are borrowed until this returns; per-archive failures are in out[i].status
    pub fn nafgpu_pipeline_wait_counts(p: *mut nafgpu_pipeline, ticket: i64, out: *mut nafgpu_counts, n: u32) -> c_int;
    /// nafgpu_job_export on the ticket's lane (after wait_counts, before release)
    pub fn nafgpu_pipeline_export(p: *mut nafgpu_pipeline, ticket: i64, spec: *const nafgpu_export, stream: *mut c_void) -> c_int;
}
