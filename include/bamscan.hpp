// bamscan.hpp -- header-only C++17 mirror of the reference's provider / execution-plan pair over the C ABI (bamscan.h).
//
// The reference's host language is Rust (BamTableProvider: datafusion/bio-format-bam/src/table_provider.rs:381-390, 928-1115;
// BamExec: physical_exec.rs:84-173); no Rust toolchain exists where this repo is built, so the compiled-language face of the
// drop-in is this header: same names, same argument order and meaning, errors as exceptions carrying bamscan_last_error()
// (the reference returns DataFusionError::Execution).  The Rust shim of INTEGRATION.md section 2 is the same code in Rust.
// Batches cross as Arrow C Data Interface structs (struct arrays whose children follow the projection order); the caller
// owns them and calls release, exactly like any other Arrow C producer.
#pragma once
#include <cstdint>
#include <cstring>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "bamscan.h"

#ifndef ARROW_C_DATA_INTERFACE
#define ARROW_C_DATA_INTERFACE
extern "C" {
struct ArrowSchema {
  const char* format; const char* name; const char* metadata; int64_t flags; int64_t n_children;
  struct ArrowSchema** children; struct ArrowSchema* dictionary; void (*release)(struct ArrowSchema*); void* private_data;
};
struct ArrowArray {
  int64_t length; int64_t null_count; int64_t offset; int64_t n_buffers; int64_t n_children; const void** buffers;
  struct ArrowArray** children; struct ArrowArray* dictionary; void (*release)(struct ArrowArray*); void* private_data;
};
}
#endif

namespace bamscan_cpp {

struct Error : std::runtime_error {
  int code;
  Error(int c, const char* msg) : std::runtime_error(msg ? msg : ""), code(c) {}
};
inline void check(int rc) { if (rc < 0) throw Error(rc, bamscan_last_error()); }

// One conjunct of `filters: &[Expr]` in the shapes the reference can push (genomic_filter.rs:151-329, record_filter.rs:285-355).
struct Filter {
  int32_t column; int32_t op;
  std::vector<double> nums; std::vector<std::string> strs;
  static Filter str(int32_t column, int32_t op, std::vector<std::string> v) { return Filter{column, op, {}, std::move(v)}; }
  static Filter num(int32_t column, int32_t op, std::vector<double> v) { return Filter{column, op, std::move(v), {}}; }
};

class FilterPack {   // keeps the C views of a filter list alive
 public:
  explicit FilterPack(const std::vector<Filter>& fs) : cstr_(fs.size()), raw_(fs.size()) {
    for (size_t i = 0; i < fs.size(); i++) {
      for (auto& s : fs[i].strs) cstr_[i].push_back(s.c_str());
      raw_[i].column = fs[i].column; raw_[i].op = fs[i].op;
      raw_[i].n_values = (int32_t)(fs[i].strs.empty() ? fs[i].nums.size() : fs[i].strs.size());
      raw_[i].num_values = fs[i].nums.empty() ? nullptr : fs[i].nums.data();
      raw_[i].str_values = cstr_[i].empty() ? nullptr : cstr_[i].data();
    }
  }
  const BamScanFilter* data() const { return raw_.empty() ? nullptr : raw_.data(); }
  int32_t size() const { return (int32_t)raw_.size(); }
 private:
  std::vector<std::vector<const char*>> cstr_;
  std::vector<BamScanFilter> raw_;
};

// == SendableRecordBatchStream of one partition (physical_exec.rs:108-172).
class RecordBatchStream {
 public:
  explicit RecordBatchStream(BamScanStream* s) : s_(s) {}
  RecordBatchStream(RecordBatchStream&& o) noexcept : s_(o.s_) { o.s_ = nullptr; }
  RecordBatchStream(const RecordBatchStream&) = delete;
  ~RecordBatchStream() { if (s_) bamscan_stream_free(s_); }
  // poll_next: true = *out holds a batch (release it), false = end of the partition; throws on a scan error.
  bool next(ArrowArray* out) { int rc = bamscan_next(s_, out); check(rc); return rc == 1; }
  BamScanStats stats() const { BamScanStats st; std::memset(&st, 0, sizeof st); check(bamscan_stream_stats(s_, &st)); return st; }
 private:
  BamScanStream* s_;
};

// == BamExec | EmptyExec (physical_exec.rs:39-56, 84-173).
class BamExec {
 public:
  explicit BamExec(BamScanPlan* p) : p_(p) {}
  BamExec(BamExec&& o) noexcept : p_(o.p_) { o.p_ = nullptr; }
  BamExec(const BamExec&) = delete;
  ~BamExec() { if (p_) bamscan_plan_free(p_); }
  int32_t output_partition_count() const { return bamscan_plan_num_partitions(p_); }   // 0 == EmptyExec
  void schema(ArrowSchema* out) const { check(bamscan_plan_schema(p_, out)); }
  RecordBatchStream execute(int32_t partition) { BamScanStream* s = nullptr; check(bamscan_execute(p_, partition, &s)); return RecordBatchStream(s); }
  int32_t num_ranges(int32_t partition) const { return bamscan_plan_num_ranges(p_, partition); }
 private:
  BamScanPlan* p_;
};

// == BamTableProvider (table_provider.rs:314-335).
class BamTableProvider {
 public:
  // == BamTableProvider::new(file_path, object_storage_options, coordinate_system_zero_based, tag_fields, binary_cigar,
  //                          infer_tag_types, infer_tag_sample_size, tag_type_hints)   (table_provider.rs:381-390)
  // object_storage_options must be empty: remote object stores are out of scope of this build (local files).
  BamTableProvider(const std::string& file_path, const std::optional<std::string>& object_storage_options = std::nullopt,
                   bool coordinate_system_zero_based = true, const std::optional<std::vector<std::string>>& tag_fields = std::nullopt,
                   bool binary_cigar = false, bool infer_tag_types = true, int32_t infer_tag_sample_size = 100,
                   const std::optional<std::vector<std::string>>& tag_type_hints = std::nullopt,
                   const std::optional<std::string>& index_path = std::nullopt, int32_t device_id = 0, int32_t batch_rows = 0) {
    if (object_storage_options) throw Error(BAMSCAN_ERR_UNSUPPORTED, "remote object storage is out of scope for this build (local files only)");
    std::vector<const char*> tags, hints;
    if (tag_fields) for (auto& t : *tag_fields) tags.push_back(t.c_str());
    if (tag_type_hints) for (auto& t : *tag_type_hints) hints.push_back(t.c_str());
    BamScanOptions o; std::memset(&o, 0, sizeof o);
    o.struct_size = sizeof o; o.coordinate_system_zero_based = coordinate_system_zero_based; o.binary_cigar = binary_cigar;
    o.has_tag_fields = tag_fields.has_value(); o.n_tag_fields = (int32_t)tags.size(); o.tag_fields = tags.empty() ? nullptr : tags.data();
    o.infer_tag_types = infer_tag_types; o.infer_tag_sample_size = infer_tag_sample_size;
    o.n_tag_type_hints = (int32_t)hints.size(); o.tag_type_hints = hints.empty() ? nullptr : hints.data();
    o.device_id = device_id; o.batch_rows = batch_rows;
    check(bamscan_open(file_path.c_str(), index_path ? index_path->c_str() : nullptr, &o, &h_));
  }
  // == try_new_with_inferred_schema (table_provider.rs:568-621)
  static BamTableProvider try_new_with_inferred_schema(const std::string& file_path, const std::optional<std::string>& object_storage_options,
                                                       bool coordinate_system_zero_based, const std::optional<std::vector<std::string>>& tag_fields,
                                                       std::optional<int32_t> sample_size, bool binary_cigar) {
    return BamTableProvider(file_path, object_storage_options, coordinate_system_zero_based, tag_fields, binary_cigar, true, sample_size.value_or(100));
  }
  BamTableProvider(BamTableProvider&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  BamTableProvider(const BamTableProvider&) = delete;
  ~BamTableProvider() { if (h_) bamscan_close(h_); }

  void schema(ArrowSchema* out) const { check(bamscan_schema(h_, out)); }                  // TableProvider::schema (:933-935)
  const char* table_type() const { return "Base"; }                                         // :937-939
  // supports_filters_pushdown (:941-962): true = Inexact, false = Unsupported
  std::vector<bool> supports_filters_pushdown(const std::vector<Filter>& filters) const {
    FilterPack fp(filters);
    std::vector<uint8_t> out(filters.size() + 1);
    check(bamscan_classify_filters(h_, fp.data(), fp.size(), out.data()));
    return std::vector<bool>(out.begin(), out.begin() + (long)filters.size());
  }
  // scan(state, projection, filters, limit) (:964-1115); target_partitions is the session's, partition_mode BAMSCAN_PARTITION_*
  BamExec scan(const std::optional<std::vector<int32_t>>& projection, const std::vector<Filter>& filters, std::optional<int64_t> limit,
               int32_t target_partitions = 1, int32_t partition_mode = BAMSCAN_PARTITION_REFERENCE) const {
    FilterPack fp(filters);
    BamScanPlan* p = nullptr;
    check(bamscan_plan(h_, projection && !projection->empty() ? projection->data() : nullptr, projection ? (int32_t)projection->size() : -1,
                       fp.data(), fp.size(), limit.value_or(-1), target_partitions, partition_mode, &p));
    return BamExec(p);
  }
  // describe (:703-927), the file-reading half: (tag, sam_type, arrow_type, description) of every aux tag in the sample, sorted
  struct TagRow { std::string tag, sam_type, arrow_type, description; };
  std::vector<TagRow> describe_tags(std::optional<int32_t> sample_size = std::nullopt) const {
    uint64_t need = 0;
    std::string buf(1 << 16, '\0');
    int rc = bamscan_describe_tags(h_, sample_size.value_or(0), buf.data(), buf.size(), &need);
    if (rc != 0 && need > buf.size()) { buf.assign(need, '\0'); rc = bamscan_describe_tags(h_, sample_size.value_or(0), buf.data(), buf.size(), &need); }
    check(rc);
    std::vector<TagRow> rows;
    size_t p = 0;
    const size_t end = std::strlen(buf.c_str());
    while (p < end) {
      size_t nl = buf.find('\n', p);
      std::string line = buf.substr(p, nl - p);
      size_t a = line.find('\t'), b = line.find('\t', a + 1), c = line.find('\t', b + 1);
      rows.push_back(TagRow{line.substr(0, a), line.substr(a + 1, b - a - 1), line.substr(b + 1, c - b - 1), line.substr(c + 1)});
      p = nl + 1;
    }
    return rows;
  }
  BamScanHandle* raw() const { return h_; }
 private:
  BamScanHandle* h_ = nullptr;
};

// == FastqTableProvider (bio-format-fastq/src/table_provider.rs:46-75, 90-151) for BGZF-compressed FASTQ: new(file_path,
// object_storage_options); scan() with BAMSCAN_PARTITION_REFERENCE follows the companion .gzi (physical_exec.rs:94-116, 140-175).
class FastqTableProvider {
 public:
  explicit FastqTableProvider(const std::string& file_path, const std::optional<std::string>& object_storage_options = std::nullopt,
                              int32_t device_id = 0, int32_t batch_rows = 0) {
    if (object_storage_options) throw Error(BAMSCAN_ERR_UNSUPPORTED, "remote object storage is out of scope for this build (local files only)");
    BamScanOptions o; std::memset(&o, 0, sizeof o);
    o.struct_size = sizeof o; o.device_id = device_id; o.batch_rows = batch_rows;
    check(bamscan_open_fastq(file_path.c_str(), &o, &h_));
  }
  FastqTableProvider(FastqTableProvider&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  FastqTableProvider(const FastqTableProvider&) = delete;
  ~FastqTableProvider() { if (h_) bamscan_close(h_); }
  void schema(ArrowSchema* out) const { check(bamscan_schema(h_, out)); }
  const char* table_type() const { return "Base"; }
  BamExec scan(const std::optional<std::vector<int32_t>>& projection, std::optional<int64_t> limit, int32_t target_partitions = 1,
               int32_t partition_mode = BAMSCAN_PARTITION_REFERENCE) const {
    BamScanPlan* p = nullptr;
    check(bamscan_plan(h_, projection && !projection->empty() ? projection->data() : nullptr, projection ? (int32_t)projection->size() : -1,
                       nullptr, 0, limit.value_or(-1), target_partitions, partition_mode, &p));
    return BamExec(p);
  }
 private:
  BamScanHandle* h_ = nullptr;
};

// A provider for BGZF-compressed FASTA (bamscan_open_fasta): name, description (nullable), sequence.  scan() with
// target_partitions > 1 cuts BGZF block ranges balanced by compressed bytes; no filter is pushed down.
class FastaTableProvider {
 public:
  explicit FastaTableProvider(const std::string& file_path, const std::optional<std::string>& object_storage_options = std::nullopt,
                              int32_t device_id = 0, int32_t batch_rows = 0) {
    if (object_storage_options) throw Error(BAMSCAN_ERR_UNSUPPORTED, "remote object storage is out of scope for this build (local files only)");
    BamScanOptions o; std::memset(&o, 0, sizeof o);
    o.struct_size = sizeof o; o.device_id = device_id; o.batch_rows = batch_rows;
    check(bamscan_open_fasta(file_path.c_str(), &o, &h_));
  }
  FastaTableProvider(FastaTableProvider&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  FastaTableProvider(const FastaTableProvider&) = delete;
  ~FastaTableProvider() { if (h_) bamscan_close(h_); }
  void schema(ArrowSchema* out) const { check(bamscan_schema(h_, out)); }
  const char* table_type() const { return "Base"; }
  BamExec scan(const std::optional<std::vector<int32_t>>& projection, std::optional<int64_t> limit, int32_t target_partitions = 1) const {
    BamScanPlan* p = nullptr;
    check(bamscan_plan(h_, projection && !projection->empty() ? projection->data() : nullptr, projection ? (int32_t)projection->size() : -1,
                       nullptr, 0, limit.value_or(-1), target_partitions,
                       target_partitions > 1 ? BAMSCAN_PARTITION_BLOCK_RANGE : BAMSCAN_PARTITION_REFERENCE, &p));
    return BamExec(p);
  }
 private:
  BamScanHandle* h_ = nullptr;
};

// == BamWriteExec (bio-format-bam/src/write_exec.rs:43-110, 195-350): INSERT OVERWRITE into a BGZF BAM.  The SAM header text and
// the reference dictionary are the caller's (the Rust host keeps build_bam_header, header_builder.rs:43-186; INTEGRATION.md 3c).
class BamWriteExec {
 public:
  BamWriteExec(const std::string& output_path, const std::string& sam_header_text, const std::vector<std::string>& ref_names,
               const std::vector<int32_t>& ref_lengths, const ArrowSchema* input_schema, const std::vector<std::string>& tag_fields = {},
               bool coordinate_system_zero_based = true, int32_t device_id = 0) {
    if (ref_names.size() != ref_lengths.size()) throw Error(BAMSCAN_ERR_INVALID, "ref_names and ref_lengths differ in length");
    std::vector<const char*> names, tags;
    for (auto& n : ref_names) names.push_back(n.c_str());
    for (auto& t : tag_fields) tags.push_back(t.c_str());
    BamWriteOptions o; std::memset(&o, 0, sizeof o);
    o.struct_size = sizeof o; o.coordinate_system_zero_based = coordinate_system_zero_based; o.device_id = device_id;
    o.n_tag_fields = (int32_t)tags.size(); o.tag_fields = tags.empty() ? nullptr : tags.data();
    check(bamscan_writer_open(output_path.c_str(), sam_header_text.c_str(), (int32_t)names.size(), names.empty() ? nullptr : names.data(),
                              ref_lengths.empty() ? nullptr : ref_lengths.data(), input_schema, &o, &w_));
  }
  BamWriteExec(BamWriteExec&& o) noexcept : w_(o.w_) { o.w_ = nullptr; }
  BamWriteExec(const BamWriteExec&) = delete;
  ~BamWriteExec() { if (w_) bamscan_writer_free(w_); }
  void write(const ArrowArray* batch) { check(bamscan_writer_write(w_, batch)); }          // one RecordBatch (struct array), not released here
  uint64_t finish() { uint64_t n = 0; check(bamscan_writer_finish(w_, &n)); return n; }    // the reference's `count`
  BamWriteStats stats() const { BamWriteStats st; std::memset(&st, 0, sizeof st); check(bamscan_writer_stats(w_, &st)); return st; }
 private:
  BamWriter* w_ = nullptr;
};

// The FASTQ write path (bamscan_fastq_writer_open): name / description / sequence / quality_scores of input_schema, looked up
// by name (description optional, other columns ignored).  compression: 0 BGZF, 1 BGZF with stored blocks, 2 plain text.
class FastqWriteExec {
 public:
  FastqWriteExec(const std::string& output_path, const ArrowSchema* input_schema, int32_t compression = 0, int32_t device_id = 0) {
    BamWriteOptions o; std::memset(&o, 0, sizeof o);
    o.struct_size = sizeof o; o.device_id = device_id; o.compression = compression;
    check(bamscan_fastq_writer_open(output_path.c_str(), input_schema, &o, &w_));
  }
  FastqWriteExec(FastqWriteExec&& o) noexcept : w_(o.w_) { o.w_ = nullptr; }
  FastqWriteExec(const FastqWriteExec&) = delete;
  ~FastqWriteExec() { if (w_) bamscan_writer_free(w_); }
  void write(const ArrowArray* batch) { check(bamscan_writer_write(w_, batch)); }          // one RecordBatch (struct array), not released here
  uint64_t finish() { uint64_t n = 0; check(bamscan_writer_finish(w_, &n)); return n; }    // rows written
  BamWriteStats stats() const { BamWriteStats st; std::memset(&st, 0, sizeof st); check(bamscan_writer_stats(w_, &st)); return st; }
 private:
  BamWriter* w_ = nullptr;
};

// The SAM write path (bamscan_sam_writer_open): BamWriteExec's arguments and row rules, written as plain SAM text -- the header
// text as given, then one line per row (no BGZF).  Rows whose line would not read back as the same row are refused (DESIGN 3.9).
class SamWriteExec {
 public:
  SamWriteExec(const std::string& output_path, const std::string& sam_header_text, const std::vector<std::string>& ref_names,
               const std::vector<int32_t>& ref_lengths, const ArrowSchema* input_schema, const std::vector<std::string>& tag_fields = {},
               bool coordinate_system_zero_based = true, int32_t device_id = 0) {
    if (ref_names.size() != ref_lengths.size()) throw Error(BAMSCAN_ERR_INVALID, "ref_names and ref_lengths differ in length");
    std::vector<const char*> names, tags;
    for (auto& n : ref_names) names.push_back(n.c_str());
    for (auto& t : tag_fields) tags.push_back(t.c_str());
    BamWriteOptions o; std::memset(&o, 0, sizeof o);
    o.struct_size = sizeof o; o.coordinate_system_zero_based = coordinate_system_zero_based; o.device_id = device_id;
    o.n_tag_fields = (int32_t)tags.size(); o.tag_fields = tags.empty() ? nullptr : tags.data();
    check(bamscan_sam_writer_open(output_path.c_str(), sam_header_text.c_str(), (int32_t)names.size(), names.empty() ? nullptr : names.data(),
                                  ref_lengths.empty() ? nullptr : ref_lengths.data(), input_schema, &o, &w_));
  }
  SamWriteExec(SamWriteExec&& o) noexcept : w_(o.w_) { o.w_ = nullptr; }
  SamWriteExec(const SamWriteExec&) = delete;
  ~SamWriteExec() { if (w_) bamscan_writer_free(w_); }
  void write(const ArrowArray* batch) { check(bamscan_writer_write(w_, batch)); }          // one RecordBatch (struct array), not released here
  uint64_t finish() { uint64_t n = 0; check(bamscan_writer_finish(w_, &n)); return n; }    // rows written
  BamWriteStats stats() const { BamWriteStats st; std::memset(&st, 0, sizeof st); check(bamscan_writer_stats(w_, &st)); return st; }
 private:
  BamWriter* w_ = nullptr;
};

}  // namespace bamscan_cpp
