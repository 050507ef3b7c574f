// bamscan_internal.h -- host-side data model shared by the planner (C++) and the device engine (CUDA).
#pragma once
#include <cstdint>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/bamscan.h"
#include "arrow_c_abi.h"

namespace bamscan {

void set_error(const char* fmt, ...);   // thread-local message for bamscan_last_error()

// column kinds (values shared with kernels_decode.cuh::ColKind)
enum : int32_t {
  HK_Int32 = 1, HK_UInt32 = 2, HK_Float32 = 3, HK_Utf8 = 4, HK_Binary = 5,
  HK_Boolean = 6,                                             // VCF Flag columns only
  HK_ListInt8 = 10, HK_ListUInt8 = 11, HK_ListInt16 = 12, HK_ListUInt16 = 13, HK_ListInt32 = 14, HK_ListUInt32 = 15, HK_ListFloat32 = 16,
  HK_ListUtf8 = 17,                                           // VCF String / Character lists only
  HK_ListListInt32 = 18, HK_ListListFloat32 = 19              // VCF FORMAT columns with Number other than 1: List<List<...>>
};

struct TagDef { std::string tag; char sam_type; int32_t kind; std::string description; };
const std::map<std::string, TagDef>& known_tags();                       // tag_registry.rs:131-684 (63 tags)
bool parse_tag_type_hints(const std::vector<std::string>& hints, std::map<std::string, std::pair<char, int32_t>>* out);   // tag_registry.rs:698-752
std::string format_sam_tag_type(char sam_type, int32_t kind);           // tag_registry.rs:65-73

struct FieldDef {
  std::string name;
  int32_t kind;
  bool nullable;
  std::vector<std::pair<std::string, std::string>> metadata;
};

struct BgzfBlock {
  uint64_t coff;        // file offset of the member
  uint32_t csize;       // total member size (BSIZE + 1)
  uint32_t cdata_off;   // offset of the deflate payload inside the member
  uint32_t isize;       // inflated size
  uint32_t crc;         // expected CRC-32
  uint64_t uoff;        // inflated offset of this member in the whole stream
};

struct BaiChunk { uint64_t beg, end; };
struct BaiRef {
  std::map<uint32_t, std::vector<BaiChunk>> bins;
  std::vector<uint64_t> intervals;            // BAI: linear index (16 KiB windows)
  std::map<uint32_t, uint64_t> loffset;       // CSI: per-bin smallest virtual offset (replaces the linear index)
  bool has_meta = false;
  uint64_t meta_beg = 0, meta_end = 0, n_mapped = 0, n_unmapped = 0;
};
// One structure for both binning indices: BAI is the fixed scheme min_shift = 14, depth = 5 (SAMv1 5.1.1); CSI carries its own
// (CSIv1 1-2).  Bin ids of level l start at (8^l - 1) / 7; the metadata pseudo-bin is first_bin(depth + 1) + 1 (37450 for BAI).
struct BaiIndex {
  std::vector<BaiRef> refs; bool has_no_coor = false; uint64_t n_no_coor = 0;
  bool csi = false; int min_shift = 14, depth = 5;
  uint32_t level_first(int l) const { return (uint32_t)(((1ull << (3 * l)) - 1) / 7); }
  uint32_t leaf_first() const { return level_first(depth); }
  uint32_t meta_bin() const { return level_first(depth + 1) + 1; }
  uint64_t max_pos() const { return 1ull << (min_shift + 3 * depth); }
};

// The file formats a scan reads (BamFile::format); the writer writes the first three
enum ScanFormat : int {
  FMT_BAM = 0,
  FMT_FASTQ = 1,   // BGZF-compressed FASTQ (kernels_fastq.cuh): same engine, four Utf8 columns, no header / index
  FMT_SAM = 2,     // plain SAM (kernels_sam.cuh): the text is transcoded to BAM records on the device, no index
  FMT_FASTA = 3,   // BGZF-compressed FASTA (kernels_fasta.cuh): three Utf8 columns, records of up to 1 GiB, no index
  FMT_VCF = 4,     // BGZF-compressed VCF (kernels_vcf.cuh): eight fixed columns and the typed INFO fields, no index
};
inline const char* format_name(int format) {
  switch (format) {
    case FMT_FASTQ: return "FASTQ";
    case FMT_SAM: return "SAM";
    case FMT_FASTA: return "FASTA";
    case FMT_VCF: return "VCF";
  }
  return "BAM";
}

// == BamTableProvider (table_provider.rs:314-335)
struct BamFile {
  int format = FMT_BAM;      // a ScanFormat; stored as int because code built against this header (the host test drivers) assigns plain integers
  std::string path, index_path;
  uint8_t* data = nullptr;   // whole file: read-only mapping (O_RDONLY / PROT_READ, not page-locked); small files: a plain copy
  uint64_t size = 0;
  bool pinned = false, mapped = false, registered = false;
  int device = 0;
  std::vector<BgzfBlock> blocks;
  uint64_t total_inflated = 0;
  // header
  std::string text;
  std::vector<std::string> ref_names;
  std::vector<int32_t> ref_lens;
  uint64_t first_record_uoff = 0;    // inflated offset of the first record
  bool header_ok = false;
  // configuration
  bool zero_based = true, binary_cigar = false, has_tag_fields = false;
  std::vector<std::string> tag_fields;
  std::vector<FieldDef> fields;      // full schema: 12 core + tag columns
  std::vector<std::pair<std::string, std::string>> schema_metadata;
  std::vector<std::string> meta_ref_names;   // from the bio.bam.reference_sequences JSON (table_provider.rs:439-444)
  std::vector<uint64_t> meta_ref_lens;
  int32_t batch_rows = 0;
  uint64_t chunk_bytes = 0;              // 0 = one inflate wave per chunk (engine.cu::plan_chunks); else the caller's cap (<= 768 MiB)
  uint32_t seg_bytes = 16384;
  bool seg_bytes_set = false;             // BamScanOptions.segment_bytes given: no adaptive segment size
  bool skip_crc = false;
  int32_t debug_flags = 0;
  bool decode_all_tags = false;           // BamScanOptions.decode_all_tag_fields
  std::unique_ptr<BaiIndex> bai;
  // VCF: the header's ##INFO lines, in header order (Number, Type and Description as written)
  struct VcfInfo { std::string id, number, type, description; };
  std::vector<VcfInfo> vcf_info;
  // VCF FORMAT: the selected IDs (BamScanOptions.format_fields; empty selects none), the ##FORMAT lines and the sample names (read
  // only when an ID is selected), and the schema index behind the last INFO column (FORMAT columns follow it)
  std::vector<std::string> format_fields;
  std::vector<VcfInfo> vcf_format;
  std::vector<std::string> vcf_samples;
  int32_t vcf_info_end = 0;
};

// genomic_filter.rs:16-32
struct GenomicRegion { std::string chrom; bool has_start = false, has_end = false; uint64_t start = 0, end = 0; bool unmapped_tail = false; };

struct RecordFilter {   // a pushed record-level predicate (record_filter.rs)
  int32_t column, op;
  std::vector<double> nums;
  std::vector<std::string> strs;
};

// One unit of device work inside a partition: a run of BGZF blocks plus the row rule to apply.
struct ScanRange {
  uint32_t block_begin = 0, block_end = 0;   // blocks whose records are owned: [block_begin, block_end)
  bool exact_start = true;                   // first_uoff is an exact record start
  uint64_t first_uoff = 0;                   // inflated offset of the first record (exact_start) / of the range start
  uint64_t stop_uoff = ~0ull;                // records starting at or after this inflated offset are not owned
  // row rule (physical_exec.rs:1036-1356); mode 0 = none (sequential full scan)
  int32_t region_mode = 0;                   // 1 mapped region, 2 per-reference unmapped tail, 3 "*" unplaced
  int32_t region_ref = -1;
  uint64_t region_start = 0, region_end = 0; // 1-based closed, 0 = open
};

struct Partition { std::vector<ScanRange> ranges; std::vector<GenomicRegion> regions; uint64_t estimated_bytes = 0; };

// == BamExec (physical_exec.rs:39-56)
struct Plan {
  BamFile* file = nullptr;
  bool has_projection = false;
  std::vector<int32_t> projection;
  std::vector<FieldDef> out_fields;
  std::vector<Partition> partitions;
  std::vector<RecordFilter> residual;
  bool empty_exec = false;
};

// host_file.cpp
int load_file(BamFile* f);                       // reads the file into pinned memory, walks BGZF, parses header
bool is_sam_path(const std::string& path);      // BamTableProvider's `is_sam`: the path ends in ".sam", any case
int load_sam(BamFile* f);                        // FMT_SAM: header lines, @SQ references, pseudo-blocks over the text body
uint64_t sam_record_start_at(const BamFile& f, uint64_t off);   // first line start at or after off (a record belongs to the range holding its first byte)
int infer_tag_types(const BamFile& f, const std::vector<std::string>& tags, int sample_size,
                    std::map<std::string, std::pair<char, int32_t>>* out, bool all = false);   // table_provider.rs:145-202
std::string discover_index(const std::string& path);   // index_utils.rs:43-76
int load_gzi(const std::string& path, std::vector<std::pair<uint64_t, uint64_t>>* out);   // bgzip -i index: (compressed, inflated) offset of every member after the first; BAMSCAN_ERR_IO when absent
int load_bai(const std::string& path, BaiIndex* out);     // BAI, or CSI when the file is BGZF / starts with "CSI\1"

// host_schema.cpp
int build_schema(BamFile* f, const BamScanOptions* opt);   // determine_schema (table_provider.rs:42-140)
int build_vcf_schema(BamFile* f, const BamScanOptions* opt);   // FMT_VCF: the eight fixed columns + the selected INFO fields
int export_schema(const std::vector<FieldDef>& fields, const std::vector<std::pair<std::string, std::string>>& metadata,
                  struct ArrowSchema* out);

// host_plan.cpp
int classify_filters(const BamFile& f, const BamScanFilter* filters, int n, uint8_t* out);
int make_plan(BamFile* f, const int32_t* projection, int32_t n_projection, const BamScanFilter* filters, int32_t n_filters,
              int32_t target_partitions, int32_t partition_mode, Plan** out);

// pinned memory helpers implemented in engine.cu (so that host .cpp files need no CUDA headers)
void* pinned_alloc(size_t bytes);
void pinned_free(void* p);
void* map_file_pinned(const char* path, uint64_t size, bool* registered);
void unmap_file_pinned(void* p, uint64_t size, bool registered);
void release_file(BamFile* f);

}  // namespace bamscan
