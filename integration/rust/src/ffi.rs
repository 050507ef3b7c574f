//! Raw bindings of `include/bamscan.h` (keep in sync with that header; every struct is `#[repr(C)]`).
#![allow(non_camel_case_types)]

use arrow::ffi::{FFI_ArrowArray, FFI_ArrowSchema};
use std::ffi::{c_char, c_int};

#[repr(C)]
pub struct BamScanHandle {
    _p: [u8; 0],
}
#[repr(C)]
pub struct BamScanPlan {
    _p: [u8; 0],
}
#[repr(C)]
pub struct BamScanStream {
    _p: [u8; 0],
}

#[repr(C)]
pub struct BamScanOptions {
    pub struct_size: u32,
    pub coordinate_system_zero_based: i32,
    pub binary_cigar: i32,
    pub has_tag_fields: i32,
    pub n_tag_fields: i32,
    pub tag_fields: *const *const c_char,
    pub infer_tag_types: i32,
    pub infer_tag_sample_size: i32,
    pub n_tag_type_hints: i32,
    pub tag_type_hints: *const *const c_char,
    pub device_id: i32,
    pub batch_rows: i32,
    pub chunk_inflated_bytes: u64,
    pub segment_bytes: u32,
    pub skip_crc: i32,
    pub debug_flags: i32,
}

#[repr(C)]
pub struct BamScanFilter {
    pub column: i32,
    pub op: i32,
    pub n_values: i32,
    pub num_values: *const f64,
    pub str_values: *const *const c_char,
}

pub const OP_EQ: i32 = 0;
pub const OP_NE: i32 = 1;
pub const OP_LT: i32 = 2;
pub const OP_LE: i32 = 3;
pub const OP_GT: i32 = 4;
pub const OP_GE: i32 = 5;
pub const OP_BETWEEN: i32 = 6;
pub const OP_NOT_BETWEEN: i32 = 7;
pub const OP_IN: i32 = 8;
pub const OP_NOT_IN: i32 = 9;
pub const OP_OTHER: i32 = 100;

pub const PUSHDOWN_UNSUPPORTED: u8 = 0;
pub const PUSHDOWN_INEXACT: u8 = 1;
pub const PARTITION_REFERENCE: i32 = 0;
pub const PARTITION_BLOCK_RANGE: i32 = 1;

unsafe extern "C" {
    pub fn bamscan_open(path: *const c_char, index_path_or_null: *const c_char, options: *const BamScanOptions, out: *mut *mut BamScanHandle) -> c_int;
    /// BGZF-compressed FASTA: the same handle and calls; schema name / description (nullable) / sequence, all Utf8.
    pub fn bamscan_open_fasta(path: *const c_char, options: *const BamScanOptions, out: *mut *mut BamScanHandle) -> c_int;
    pub fn bamscan_close(h: *mut BamScanHandle);
    pub fn bamscan_schema(h: *mut BamScanHandle, out: *mut FFI_ArrowSchema) -> c_int;
    /// describe(): "TAG\tsam_type\tarrow_type\tdescription\n" per aux tag of the first `sample_size` records.
    pub fn bamscan_describe_tags(h: *mut BamScanHandle, sample_size: i32, buf: *mut std::os::raw::c_char, cap: u64, needed: *mut u64) -> c_int;
    pub fn bamscan_classify_filters(h: *mut BamScanHandle, filters: *const BamScanFilter, n: i32, out_pushdown: *mut u8) -> c_int;
    pub fn bamscan_plan(
        h: *mut BamScanHandle,
        projection: *const i32,
        n_projection: i32,
        filters: *const BamScanFilter,
        n_filters: i32,
        limit_or_neg: i64,
        target_partitions: i32,
        partition_mode: i32,
        out: *mut *mut BamScanPlan,
    ) -> c_int;
    pub fn bamscan_plan_num_partitions(p: *const BamScanPlan) -> i32;
    pub fn bamscan_plan_schema(p: *const BamScanPlan, out: *mut FFI_ArrowSchema) -> c_int;
    pub fn bamscan_plan_free(p: *mut BamScanPlan);
    pub fn bamscan_execute(p: *mut BamScanPlan, partition: i32, out: *mut *mut BamScanStream) -> c_int;
    pub fn bamscan_next(s: *mut BamScanStream, out: *mut FFI_ArrowArray) -> c_int;
    pub fn bamscan_stream_free(s: *mut BamScanStream);
    pub fn bamscan_last_error() -> *const c_char;

    // write path (INSERT OVERWRITE): include/bamscan.h, "SURVEY 8 f4"
    pub fn bamscan_writer_open(
        output_path: *const c_char,
        sam_header_text: *const c_char,
        n_ref: i32,
        ref_names: *const *const c_char,
        ref_lengths: *const i32,
        input_schema: *const FFI_ArrowSchema,
        options: *const BamWriteOptions,
        out: *mut *mut BamWriter,
    ) -> c_int;
    pub fn bamscan_writer_write(w: *mut BamWriter, batch: *const FFI_ArrowArray) -> c_int;
    pub fn bamscan_writer_finish(w: *mut BamWriter, rows_written: *mut u64) -> c_int;
    pub fn bamscan_writer_free(w: *mut BamWriter);
    // FASTQ write path: the same BamWriter handle and calls; options read: struct_size, device_id, compression (0/1 BGZF, 2 plain)
    pub fn bamscan_fastq_writer_open(
        output_path: *const c_char,
        input_schema: *const FFI_ArrowSchema,
        options: *const BamWriteOptions,
        out: *mut *mut BamWriter,
    ) -> c_int;
    // SAM write path: bamscan_writer_open's arguments, plain SAM text (header text as given, one line per row); compression not read
    pub fn bamscan_sam_writer_open(
        output_path: *const c_char,
        sam_header_text: *const c_char,
        n_ref: i32,
        ref_names: *const *const c_char,
        ref_lengths: *const i32,
        input_schema: *const FFI_ArrowSchema,
        options: *const BamWriteOptions,
        out: *mut *mut BamWriter,
    ) -> c_int;
}

#[repr(C)]
pub struct BamWriter {
    _p: [u8; 0],
}

/// == BamWriteOptions of include/bamscan.h (zero-initialise, set struct_size)
#[repr(C)]
pub struct BamWriteOptions {
    pub struct_size: u32,
    pub coordinate_system_zero_based: i32,
    pub n_tag_fields: i32,
    pub tag_fields: *const *const c_char,
    pub device_id: i32,
    pub compression: i32,
}
