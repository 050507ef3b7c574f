/*
 * bamscan.h -- C ABI of the B200-native BAM table scan (libbamscan.so).
 *
 * This is the drop-in boundary for ONE path of biodatageeks/datafusion-bio-formats: the local-file
 * `SELECT ... FROM bam` scan, `BamTableProvider::scan -> BamExec::execute`.  Each entry point names the
 * reference interface it replaces (paths relative to the reference repository root).  Everything that
 * crosses is POD or the Arrow C Data Interface (struct ArrowSchema / struct ArrowArray); there are no
 * CUDA, torch or C++ types in any signature.  Batches come back in host memory, ready for
 * `arrow::ffi::from_ffi` (Rust) / `pyarrow.RecordBatch._import_from_c` (Python).
 *
 * There is no CPU fallback inside the library: bamscan_execute / bamscan_run_device_resident fail with
 * BAMSCAN_ERR_CUDA when no device is present.  Planning calls (open, schema, classify_filters, plan) are host-only,
 * like the reference's provider construction and `scan()`, and work anywhere.
 *
 * Threading: handles are not thread-safe individually; distinct streams may be driven from distinct
 * host threads (the reference's "one thread per partition", bio-format-core/src/sync_stream.rs:7-33).
 */
#ifndef BAMSCAN_H
#define BAMSCAN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

struct ArrowSchema;
struct ArrowArray;

typedef struct BamScanHandle BamScanHandle;   /* an opened BAM  == BamTableProvider          */
typedef struct BamScanPlan BamScanPlan;       /* a planned scan == Arc<dyn ExecutionPlan> (BamExec | EmptyExec) */
typedef struct BamScanStream BamScanStream;   /* one partition  == SendableRecordBatchStream */

/* return codes: 0 ok, negative error class; message via bamscan_last_error() */
enum {
  BAMSCAN_OK = 0,
  BAMSCAN_ERR_IO = -1,           /* open/read failure                                   */
  BAMSCAN_ERR_FORMAT = -2,       /* not BGZF/BAM, corrupt record chain, bad aux         */
  BAMSCAN_ERR_CRC = -3,          /* BGZF CRC32 / ISIZE / DEFLATE stream error           */
  BAMSCAN_ERR_CUDA = -4,         /* no device, allocation or launch failure             */
  BAMSCAN_ERR_UNSUPPORTED = -5,  /* an unpinned edge this build refuses (DESIGN.md)     */
  BAMSCAN_ERR_INVALID = -6,      /* bad argument / configuration                        */
  BAMSCAN_ERR_SCHEMA = -7        /* tag value does not fit the column type (ArrowError::SchemaError in the reference) */
};

/*
 * Options == the constructor arguments of the reference provider
 *   BamTableProvider::new(file_path, object_storage_options, coordinate_system_zero_based, tag_fields,
 *                         binary_cigar, infer_tag_types, infer_tag_sample_size, tag_type_hints)
 *   (datafusion/bio-format-bam/src/table_provider.rs:381-390)
 * plus the DataFusion SessionConfig knobs the scan reads (batch_size: physical_exec.rs:129) and device
 * placement.  Zero-initialise, set struct_size = sizeof(BamScanOptions).
 */
typedef struct BamScanOptions {
  uint32_t struct_size;
  int32_t coordinate_system_zero_based;   /* table_provider.rs:384 */
  int32_t binary_cigar;                   /* table_provider.rs:386 */
  int32_t has_tag_fields;                 /* 0 => tag_fields = None */
  int32_t n_tag_fields;
  const char* const* tag_fields;          /* table_provider.rs:385 */
  int32_t infer_tag_types;                /* table_provider.rs:387 */
  int32_t infer_tag_sample_size;          /* table_provider.rs:388 */
  int32_t n_tag_type_hints;
  const char* const* tag_type_hints;      /* "TAG:TYPE" | "TAG:B:SUBTYPE", tag_registry.rs:698-752 */
  int32_t device_id;                      /* CUDA device ordinal for this handle */
  int32_t batch_rows;                     /* rows per emitted batch; 0 = one batch per device chunk (reference default 8192) */
  uint64_t chunk_inflated_bytes;          /* device chunk size cap (inflated bytes), max 768 MiB; 0 = one inflate wave per chunk (~1.5 GiB on a B200), decoded in slices of <= 768 MiB: one batch per slice */
  uint32_t segment_bytes;                 /* record-boundary segment size; 0 = default 16 KiB */
  int32_t skip_crc;                       /* 0 (default): verify CRC32 of every BGZF member on the device; 1: skip */
  int32_t debug_flags;                    /* tests only. bit0: poison boundary candidates (exercises the repair path); bit1: force the long-record decode kernels (a warp per record); bit2 / bit3 / bit4: force the warp-per-member / the lane-group / the CTA-per-member inflate kernel (default: the CTA-per-member kernel); bit5: queue the next chunk's inflate behind the current chunk's first decode slice (the two overlap on the GPU; measured +1 % scan rate, -10 % inflate rate); bit6: skip the parallel boundary-repair rounds (every disagreeing seam goes to the sequential repair) */
  int32_t decode_all_tag_fields;          /* 1: reference behaviour (sam_tag_io.rs:42-52): once ANY tag column is projected every tag_fields entry is decoded, so a value that does not fit an UNPROJECTED tag column's type fails the scan; 0 (default): only projected tag columns are decoded */
} BamScanOptions;

/* ---- pushed-down predicates (reference: `filters: &[Expr]` of TableProvider::scan, restricted to the
 * shapes the reference can push: genomic_filter.rs:151-329 and record_filter.rs:285-355) ---- */
enum { BAMSCAN_COL_NAME = 0, BAMSCAN_COL_CHROM = 1, BAMSCAN_COL_START = 2, BAMSCAN_COL_END = 3, BAMSCAN_COL_FLAGS = 4,
       BAMSCAN_COL_CIGAR = 5, BAMSCAN_COL_MAPQ = 6, BAMSCAN_COL_MATE_CHROM = 7, BAMSCAN_COL_MATE_START = 8,
       BAMSCAN_COL_SEQUENCE = 9, BAMSCAN_COL_QUALITY = 10, BAMSCAN_COL_TLEN = 11 };
enum { BAMSCAN_OP_EQ = 0, BAMSCAN_OP_NE = 1, BAMSCAN_OP_LT = 2, BAMSCAN_OP_LE = 3, BAMSCAN_OP_GT = 4, BAMSCAN_OP_GE = 5,
       BAMSCAN_OP_BETWEEN = 6, BAMSCAN_OP_NOT_BETWEEN = 7, BAMSCAN_OP_IN = 8, BAMSCAN_OP_NOT_IN = 9,
       BAMSCAN_OP_OTHER = 100 /* any expression shape the reference cannot push (OR, functions, ...) */ };
typedef struct BamScanFilter {
  int32_t column;                 /* schema index (BAMSCAN_COL_* or >= 12 for a tag column) */
  int32_t op;
  int32_t n_values;
  const double* num_values;       /* numeric literals (EQ..GE: 1, BETWEEN: 2, IN: n) or NULL */
  const char* const* str_values;  /* string literals for Utf8 columns or NULL */
} BamScanFilter;
enum { BAMSCAN_PUSHDOWN_UNSUPPORTED = 0, BAMSCAN_PUSHDOWN_INEXACT = 1 };

/* ---- partitioning ---- */
enum {
  BAMSCAN_PARTITION_REFERENCE = 0,   /* the reference's rule: no index -> 1 partition; index -> <= target_partitions
                                        balanced region partitions (table_provider.rs:1036-1114).  FASTQ handles: a
                                        companion `<path>.gzi` -> min(target, blocks) runs of whole BGZF blocks cut by
                                        block count (bio-format-fastq physical_exec.rs:94-116, 140-175), else 1 partition */
  BAMSCAN_PARTITION_BLOCK_RANGE = 1  /* target_partitions contiguous BGZF block ranges (multi-GPU full scans);
                                        concatenated in partition order the rows equal the 1-partition scan */
};

struct BamScanAssignedRegion;
typedef struct BamScanStats {
  uint64_t rows, batches, chunks;
  uint64_t compressed_bytes, inflated_bytes, arrow_bytes;   /* B_comp, B_inflated, B_arrow (SURVEY 8d) */
  uint64_t h2d_bytes, d2h_bytes;
  uint64_t blocks, kernel_launches, boundary_repairs;
  double ms_total, ms_inflate, ms_boundary, ms_decode;      /* CUDA-event device times.  Plain SAM (no inflate): compressed_bytes ==
                                                             * inflated_bytes == text bytes, ms_inflate is the ingest copy of the
                                                             * text, ms_boundary the line framing plus the SAM -> BAM transcode */
  uint64_t boundary_seam_mismatches;                        /* seams the parallel check rejected (each triggers the repair walk) */
  /* Block-range partitions: inflated offset of the first record this partition owned (UINT64_MAX: none) and the offset at
   * which its record chain landed at or after its stop offset.  Partition p > 0 SPECULATES its first record; the scan of the
   * whole file is proven exact when end_chain_uoff of partition p - 1 equals first_record_uoff of partition p for every p
   * (bamscan_check_partition_seams; the python mirror and bench.py do this and fail loudly otherwise). */
  uint64_t first_record_uoff, end_chain_uoff;
  /* BGZF members the CTA-per-member inflate kernel refused (a Huffman code whose second-level tables exceed its shared-memory
   * budget) and the warp-per-member kernel then inflated. */
  uint64_t inflate_retries;
} BamScanStats;

/* Seam check over the stats of the N block-range partitions of one plan, in partition order.  0 = every partition starts
 * where its predecessor's chain landed; BAMSCAN_ERR_FORMAT (message names the partition) otherwise. */
int bamscan_check_partition_seams(const BamScanStats* stats, int32_t n_partitions);

/* == BamTableProvider::new (table_provider.rs:381-529): header read, tag-type inference, schema, index discovery.
 * A path ending in ".sam" (any case) is read as plain SAM text, as the reference's `is_sam` does: header = the leading '@'
 * lines (references from @SQ SN / LN), each line transcoded to a BAM record on the device, the same columns; no index is
 * discovered or read.  A ".sam" file that starts with the gzip magic is refused with BAMSCAN_ERR_UNSUPPORTED.
 * index_path_or_null: NULL => discover `<path>.bai`, `<stem>.bai`, then `<path>.csi` (index_utils.rs:43-76); a BAI or a CSI
 *   (CSIv1, BGZF or plain, any min_shift / depth up to 9 levels) is read -- the reference discovers a CSI but parses it as a BAI;
 * "" => behave as if no index existed (sequential single-partition scans). */
int bamscan_open(const char* path, const char* index_path_or_null, const BamScanOptions* options, BamScanHandle** out);

/* == BamTableProvider::describe (table_provider.rs:703-927), the part that reads the file: every aux tag present in the first
 * `sample_size` records (<= 0: 100), first occurrence deciding its type (infer_type_from_noodles_value, tag_registry.rs:772-792),
 * sorted by name, one line per tag "TAG\tsam_type\tarrow_type\tdescription\n" (description: the registry's, else
 * "Custom/unknown tag (<sam_type>)"), NUL-terminated into buf.  *needed = bytes required; BAMSCAN_ERR_INVALID when cap is smaller
 * (call again).  The twelve core rows of describe() are constants the binding adds (python: BamTableProvider.describe). */
int bamscan_describe_tags(BamScanHandle* h, int32_t sample_size, char* buf, uint64_t cap, uint64_t* needed);
void bamscan_close(BamScanHandle* h);

/* == FastqTableProvider::new (bio-format-fastq/src/table_provider.rs:63-75) for a BGZF-compressed FASTQ file (SURVEY 8 f3).
 * The handle is used with the same calls as a BAM handle: bamscan_schema gives determine_schema (table_provider.rs:22-32:
 * name, description (nullable), sequence, quality_scores, all Utf8); bamscan_plan with BAMSCAN_PARTITION_BLOCK_RANGE cuts the
 * BGZF block table as get_bgzf_partition_bounds does (physical_exec.rs:140-175; a partition > 0 finds its first record by
 * the '@' ... '+' rule of synchronize_bgzf_reader, :184-219, and the seam check proves it); bamscan_execute / bamscan_next
 * (and the device variants) stream the batches of physical_exec.rs:393-468.  No filter is pushed down (classify: all
 * unsupported), there is no index, the options that concern BAM columns are ignored.  Plain gzip and uncompressed FASTQ are
 * refused (BAMSCAN_ERR_FORMAT): this build reads BGZF. */
int bamscan_open_fastq(const char* path, const BamScanOptions* options, BamScanHandle** out);

/* A BGZF-compressed FASTA file (a provider like bio-format-fasta's).  The handle is used with the same calls as a FASTQ handle:
 * bamscan_schema gives name (Utf8), description (Utf8, nullable) and sequence (Utf8).  A record is a line that starts with '>'
 * (its text up to the line end, without one trailing '\r', split at the first space or tab into name and description; an empty
 * description is NULL) followed by every line up to the next '>' line or the end of the file, joined without their line breaks
 * (and one trailing '\r' each); bytes are kept as given.  bamscan_plan with BAMSCAN_PARTITION_BLOCK_RANGE balances BGZF block
 * ranges by compressed bytes (a record belongs to the range that holds its '>'); otherwise one partition.  BAMSCAN_ERR_FORMAT,
 * naming the record of the partition: an empty name, a byte of 0x80 or above in a projected column, bytes other than whitespace in
 * front of the first '>'.  A record of more than 1 GiB of text is BAMSCAN_ERR_UNSUPPORTED.  No filter is pushed down, there is
 * no index, describe is refused, the options that concern BAM columns are ignored.  Plain gzip and uncompressed FASTA are
 * refused (BAMSCAN_ERR_FORMAT): this build reads BGZF. */
int bamscan_open_fasta(const char* path, const BamScanOptions* options, BamScanHandle** out);

/* == TableProvider::schema (table_provider.rs:933-935): the full, unprojected schema with all metadata. */
int bamscan_schema(BamScanHandle* h, struct ArrowSchema* out);

/* == TableProvider::supports_filters_pushdown (table_provider.rs:941-962). */
int bamscan_classify_filters(BamScanHandle* h, const BamScanFilter* filters, int32_t n_filters, uint8_t* out_pushdown);

/* == TableProvider::scan (table_provider.rs:964-1115).  n_projection < 0 => projection None (all columns);
 * 0 => empty projection (row counts only).  `limit` is accepted and ignored like the reference (physical_exec.rs:44). */
int bamscan_plan(BamScanHandle* h, const int32_t* projection, int32_t n_projection, const BamScanFilter* filters,
                 int32_t n_filters, int64_t limit_or_neg, int32_t target_partitions, int32_t partition_mode, BamScanPlan** out);
int32_t bamscan_plan_num_partitions(const BamScanPlan* plan);   /* == output_partitioning().partition_count(); 0 => EmptyExec */
int bamscan_plan_schema(const BamScanPlan* plan, struct ArrowSchema* out);   /* == ExecutionPlan::schema (projected) */
void bamscan_plan_free(BamScanPlan* plan);
/* Introspection of a partition's device work (== BamExec::partition_assignments, physical_exec.rs:52): number of block
 * ranges and, per range, out[14] = { block_begin, block_end, compressed offset of block_begin, compressed offset of
 * block_end, exact_start, first inflated offset, stop inflated offset (~0 = none), region_mode (0 none, 1 mapped region,
 * 2 per-reference unmapped tail, 3 "*" unplaced), region_ref, region_start, region_end (1-based closed, 0 = open),
 * partition estimated bytes, start virtual offset, stop virtual offset (0 = none) }. */
int32_t bamscan_plan_num_ranges(const BamScanPlan* plan, int32_t partition);
int bamscan_plan_range_info(const BamScanPlan* plan, int32_t partition, int32_t range, uint64_t out[14]);
/* The GenomicRegions assigned to a partition (== PartitionAssignment::regions): returns the count; fills up to `cap`
 * entries (estimate_index = reference id of the region's chromosome, -1 for "*" / unknown names). */
int32_t bamscan_plan_partition_regions(const BamScanPlan* plan, int32_t partition, struct BamScanAssignedRegion* out, int32_t cap);

/* == extract_genomic_regions (bio-format-core/src/genomic_filter.rs:51-100): the conjunction of `filters` reduced to
 * chromosomes + one [start, end] window in 1-based closed coordinates.  `chroms` holds n_chroms NUL-terminated names,
 * sorted and de-duplicated; bit i of residual_mask is set when filter i was NOT consumed as a genomic constraint. */
typedef struct BamScanRegionAnalysis {
  int32_t unsatisfiable, has_start, has_end, n_chroms;
  uint64_t start, end, residual_mask;
  char chroms[4096];
} BamScanRegionAnalysis;
int bamscan_extract_regions(const BamScanFilter* filters, int32_t n_filters, int32_t coordinate_system_zero_based,
                            BamScanRegionAnalysis* out);

/* == balance_partitions (bio-format-core/src/partition_balancer.rs:15-41, 61-295).  Input = RegionSizeEstimate[],
 * output = the regions of every PartitionAssignment, flattened in partition order (estimate_index says which input
 * estimate a (sub-)region came from). */
typedef struct BamScanRegionEstimate {
  const char* chrom;
  int32_t has_start, has_end;
  uint64_t start, end;                 /* 1-based closed */
  uint64_t estimated_bytes;
  uint64_t contig_length;              /* 0 = None */
  uint64_t unmapped_count;
  const uint64_t* nonempty_bin_positions;
  int32_t n_bin_positions;
  uint64_t leaf_bin_span;
} BamScanRegionEstimate;
typedef struct BamScanAssignedRegion {
  int32_t partition, estimate_index;
  int32_t has_start, has_end;
  uint64_t start, end;
  int32_t unmapped_tail;
  uint64_t partition_total_estimated_bytes;
} BamScanAssignedRegion;
int bamscan_balance_partitions(const BamScanRegionEstimate* estimates, int32_t n, int32_t target_partitions,
                               BamScanAssignedRegion* out, int32_t cap, int32_t* n_out, int32_t* n_partitions);

/* == ExecutionPlan::execute(partition, ctx) (physical_exec.rs:108-172). */
int bamscan_execute(BamScanPlan* plan, int32_t partition, BamScanStream** out);
/* == Stream::poll_next: 1 = a batch was written to *out (struct array, children in projection order),
 * 0 = end of stream, < 0 = error (DataFusionError::Execution in the reference, physical_exec.rs:567-571). */
int bamscan_next(BamScanStream* s, struct ArrowArray* out);

/* SURVEY 8 f2 -- device-resident hand-off for GPU consumers (no reference counterpart: the reference has no device path).
 * Same contract as bamscan_execute / bamscan_next, but the batch stays in HBM: the struct array's buffers are device
 * pointers into one allocation owned by the batch (released by the consumer through ArrowArray::release), exported with
 * the Arrow C Device Data Interface (device_type ARROW_DEVICE_CUDA, device_id, sync_event = cudaEvent_t* to wait on).
 * null_count is -1 (unknown) for nullable columns.  The 42 GB of Arrow D2H per 100 M reads disappear for such consumers. */
struct ArrowDeviceArray;
int bamscan_execute_device(BamScanPlan* plan, int32_t partition, BamScanStream** out);
int bamscan_next_device(BamScanStream* stream, struct ArrowDeviceArray* out);
void bamscan_stream_free(BamScanStream* s);

/* ---- measurement hooks (bench.py only) ---- */
/* Stages the partition's compressed bytes in HBM before the clock starts and keeps every Arrow buffer in HBM
 * (no H2D / D2H inside the scan); runs the whole partition and fills *stats.  Used for the device-resident
 * `value` of bench.py; the product path is bamscan_execute/bamscan_next. */
int bamscan_run_device_resident(BamScanPlan* plan, int32_t partition, int32_t repeats, BamScanStats* stats);
int bamscan_stream_stats(const BamScanStream* s, BamScanStats* out);
/* Inflate-only microbenchmark on the partition's blocks (roofline of the dominant kernel): device ms per launch. */
int bamscan_bench_inflate(BamScanPlan* plan, int32_t partition, int32_t repeats, double* ms_per_launch, uint64_t* inflated_bytes,
                          uint64_t* compressed_bytes);

/* Pinned-memory PCIe probe (the end-to-end ceiling): best of 3 for H2D, D2H and both at once, GB/s. */
int bamscan_probe_pcie(int32_t device_id, uint64_t bytes, double* h2d_gbps, double* d2h_gbps, double* bidir_gbps);


/* ---- SURVEY 8 f4: the BAM WRITE path (`INSERT OVERWRITE INTO bam_table SELECT ...`) --------------------------------
 * == BamTableProvider::insert_into -> BamWriteExec::execute -> write_bam_stream
 *    (datafusion/bio-format-bam/src/table_provider.rs:1117-1177, write_exec.rs:195-350), with
 *    batch_to_alignment_records (bio-format-core/src/sam_record_serializer.rs:15-212), build_tag_data
 *    (bio-format-core/src/sam_tag_io.rs:109-147) and the noodles BAM record encoder + BGZF writer on the device:
 *    Arrow batches (host memory, Arrow C Data Interface) -> H2D -> BAM records encoded by CUDA kernels -> BGZF members of
 *    0xff00 inflated bytes compressed by a CTA-per-member DEFLATE kernel (LZ77 + dynamic Huffman, CRC-32 fused) -> D2H ->
 *    file.  The SAM header text and the reference dictionary come from the caller: the Rust host keeps build_bam_header
 *    (header_builder.rs:43-186) and serialises its result (INTEGRATION.md 3c); the python mirror restates it.
 *    `input_schema` names the columns (the reference looks every column up BY NAME: name, chrom, start, flags, cigar (Utf8 or
 *    Binary), mapping_quality, mate_chrom, mate_start, sequence, quality_scores, template_length) and carries the tag
 *    columns' field metadata (bio.bam.tag.tag / bio.bam.tag.type decide the aux type letter, sam_tag_io.rs:127-141).
 *    Tag columns may be integers of 8 to 64 bits, Float32 / Float64, Utf8 or List<Int8..UInt32 | Float32> (what the scan produces
 *    and what a query can make of it); other Arrow types are refused with BAMSCAN_ERR_UNSUPPORTED, as are records with more than
 *    65535 CIGAR ops (CG-tag overflow).
 *    Rows are written in arrival order (sort_on_write is a DataFusion SortExec in front of the writer, not part of it).
 *    Data errors of the reference ("does not fit into 16-bit SAM flags", CIGAR parse errors, tag range / type mismatches,
 *    sequence / quality length mismatch) come back as BAMSCAN_ERR_FORMAT / BAMSCAN_ERR_SCHEMA with the row in the message. */
typedef struct BamWriter BamWriter;
typedef struct BamWriteOptions {
  uint32_t struct_size;
  int32_t coordinate_system_zero_based;   /* write_exec.rs:208 */
  int32_t n_tag_fields;
  const char* const* tag_fields;          /* write_exec.rs:207; aux fields are written in this order */
  int32_t device_id;
  int32_t compression;                    /* 0 (default): LZ77 + dynamic Huffman; 1: stored DEFLATE blocks (tests) */
} BamWriteOptions;
typedef struct BamWriteStats {
  uint64_t rows, batches, members;
  uint64_t arrow_bytes, bam_bytes, compressed_bytes;   /* H2D Arrow bytes, uncompressed BAM stream bytes, file bytes */
  double ms_encode, ms_deflate, ms_total;               /* CUDA-event device times */
  uint64_t kernel_launches;
} BamWriteStats;
int bamscan_writer_open(const char* output_path, const char* sam_header_text, int32_t n_ref, const char* const* ref_names,
                        const int32_t* ref_lengths, const struct ArrowSchema* input_schema, const BamWriteOptions* options,
                        BamWriter** out);
/* One RecordBatch as a struct array matching input_schema (not released by the callee). */
int bamscan_writer_write(BamWriter* w, const struct ArrowArray* batch);
/* The same for a batch that lives in HBM on the writer's device (Arrow C Device Data Interface, e.g. what bamscan_next_device
 * hands out, or a GPU consumer's filtered copy of it): no H2D, the encoder reads the batch's buffers in place; waits for
 * batch->sync_event.  Not released by the callee. */
int bamscan_writer_write_device(BamWriter* w, const struct ArrowDeviceArray* batch);
/* Flushes the last (partial) member and the BGZF EOF marker, closes the file; *rows_written = the reference's `count`. */
int bamscan_writer_finish(BamWriter* w, uint64_t* rows_written);
int bamscan_writer_stats(const BamWriter* w, BamWriteStats* out);
void bamscan_writer_free(BamWriter* w);

/* ---- the FASTQ write path: Arrow batches -> FASTQ text encoded on the device -> BGZF members (or plain text) -> file ----
 * Opens a writer whose handle works with bamscan_writer_write, _write_device, _finish, _stats and _free exactly as above.
 * `input_schema` columns are looked up BY NAME: name, sequence and quality_scores are required, description is optional, all
 * Utf8; other columns are ignored, so a BAM scan's batch can be written as FASTQ too (its bases and qualities are written as
 * stored: reverse-strand reads are NOT reverse-complemented).  Schema errors (BAMSCAN_ERR_SCHEMA) come before the device is
 * touched; without a device the call fails with BAMSCAN_ERR_CUDA and creates no file.
 * Options read: struct_size, device_id, compression -- 0 (default) BGZF with LZ77 + dynamic Huffman, 1 BGZF with stored
 * blocks, 2 plain text (no BGZF, no EOF marker; accepted by FASTQ writers only).  BGZF members hold 0xff00 bytes of text, the
 * file ends with the BGZF EOF marker.
 * Each row is written as '@' name [' ' description] '\n' sequence '\n' '+' '\n' quality '\n'; the description and its separator
 * are left out when it is NULL or empty.  Bytes are written as given (no case folding, sequence and quality lengths are not
 * compared).  A NULL name / sequence / quality, a '\n' or '\r' in any field, or a space or tab in the name (the file would not
 * read back as the same rows) is BAMSCAN_ERR_FORMAT with the row in the message.
 * BamWriteStats of a FASTQ writer: bam_bytes = uncompressed FASTQ text bytes; members and ms_deflate are 0 in plain mode. */
int bamscan_fastq_writer_open(const char* output_path, const struct ArrowSchema* input_schema, const BamWriteOptions* options,
                              BamWriter** out);

/* ---- the SAM write path: Arrow batches -> SAM text lines encoded on the device -> plain text file ----
 * Arguments, schema checks and tag handling are bamscan_writer_open's, and the handle works with bamscan_writer_write,
 * _write_device, _finish, _stats and _free exactly as above.  The file starts with sam_header_text as given (the text passed to
 * bamscan_writer_open); each row becomes one line, in arrival order; there is no BGZF and no EOF marker; zero rows leave the
 * header alone.  Options read: struct_size, coordinate_system_zero_based, n_tag_fields, tag_fields, device_id (`compression` is
 * not read: BGZF-compressed SAM is not built).
 * A row is accepted or refused exactly as bamscan_writer_open's writer would, with the same error class and reason; on top of
 * that a row whose line would not read back as the same row is BAMSCAN_ERR_FORMAT with the row in the message: a name outside
 * SAMv1 [!-?A-~]{1,254} (NULL or "*" write '*'), a sequence outside [A-Za-z=.] (written as given, no case folding), a quality
 * character above '~' (characters below '!' are written as '!'), a Z value outside [ !-~], an A value outside [!-~].
 * A tag column named outside [A-Za-z][A-Za-z0-9] is BAMSCAN_ERR_SCHEMA before the device is touched.
 * Fields: RNAME / RNEXT are the resolved reference's name, '*' for none, RNEXT '=' for the record's own reference; POS / PNEXT
 * are 1-based, 0 when missing; CIGAR is rendered from its parsed operations ('*' for none); integer tags are written as
 * TG:i:<decimal>, f values as Rust's f32 Display prints them (NaN, inf, -inf), H values upper-cased (DESIGN 3.9).
 * BamWriteStats of a SAM writer: bam_bytes = SAM text bytes (header included) = compressed_bytes; members and ms_deflate are 0. */
int bamscan_sam_writer_open(const char* output_path, const char* sam_header_text, int32_t n_ref, const char* const* ref_names,
                            const int32_t* ref_lengths, const struct ArrowSchema* input_schema, const BamWriteOptions* options,
                            BamWriter** out);

const char* bamscan_last_error(void);   /* thread-local message of the last failing call on this thread */
const char* bamscan_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BAMSCAN_H */
