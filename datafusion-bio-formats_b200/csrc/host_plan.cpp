// host_plan.cpp -- scan planning: projection, filter classification, partitions.
//
// Replaces (reference, datafusion/):
//   bio-format-bam/src/table_provider.rs:941-962   supports_filters_pushdown
//   bio-format-bam/src/table_provider.rs:964-1115  scan(): projected schema, regions, partitions, residual filters
//   bio-format-core/src/genomic_filter.rs:51-329   Expr -> genomic regions          (host_index.cpp)
//   bio-format-core/src/partition_balancer.rs:61-295 balance_partitions             (host_index.cpp)
//   bio-format-bam/src/storage.rs:336-450          BAI size estimates               (host_index.cpp)
// plus the block-range partitioner of the B200 build (BASELINE north_star item 5; pattern:
// bio-format-fastq/src/physical_exec.rs:140-175 get_bgzf_partition_bounds).
#include <algorithm>
#include <cstring>

#include "bamscan_internal.h"

namespace bamscan {

int plan_indexed(BamFile* f, Plan* plan, const BamScanFilter* filters, int32_t n_filters, int32_t target_partitions, bool* handled);   // host_index.cpp

static bool is_numeric_kind(int32_t k) { return k == HK_UInt32 || k == HK_Int32 || k == HK_Float32; }

// record_filter.rs:285-355 -- which single-column comparisons can be evaluated at record level
static bool can_push_record_filter(const BamFile& f, const BamScanFilter& flt) {
  if (flt.column < 0 || flt.column >= (int32_t)f.fields.size()) return false;
  int32_t kind = f.fields[flt.column].kind;
  bool numeric_lits = flt.num_values != nullptr, string_lits = flt.str_values != nullptr;
  switch (flt.op) {
    case BAMSCAN_OP_EQ: case BAMSCAN_OP_NE:
      return (kind == HK_Utf8 && (string_lits || numeric_lits)) || (is_numeric_kind(kind) && (numeric_lits || string_lits));
    case BAMSCAN_OP_LT: case BAMSCAN_OP_LE: case BAMSCAN_OP_GT: case BAMSCAN_OP_GE:
      return is_numeric_kind(kind);
    case BAMSCAN_OP_BETWEEN: case BAMSCAN_OP_NOT_BETWEEN:
      return is_numeric_kind(kind);
    case BAMSCAN_OP_IN: case BAMSCAN_OP_NOT_IN:
      return kind == HK_Utf8 || is_numeric_kind(kind);
    default: return false;
  }
}

// genomic_filter.rs:120-148
static bool is_genomic_coordinate_filter(const BamScanFilter& flt) {
  switch (flt.op) {
    case BAMSCAN_OP_EQ: case BAMSCAN_OP_NE: case BAMSCAN_OP_LT: case BAMSCAN_OP_LE: case BAMSCAN_OP_GT: case BAMSCAN_OP_GE:
      return flt.column == BAMSCAN_COL_CHROM || flt.column == BAMSCAN_COL_START || flt.column == BAMSCAN_COL_END;
    case BAMSCAN_OP_BETWEEN: case BAMSCAN_OP_NOT_BETWEEN:
      return flt.column == BAMSCAN_COL_START || flt.column == BAMSCAN_COL_END;
    case BAMSCAN_OP_IN: case BAMSCAN_OP_NOT_IN:
      return flt.column == BAMSCAN_COL_CHROM;
    default: return false;
  }
}

int classify_filters(const BamFile& f, const BamScanFilter* filters, int n, uint8_t* out) {
  for (int i = 0; i < n; i++) {
    if (!f.index_path.empty() && is_genomic_coordinate_filter(filters[i])) out[i] = BAMSCAN_PUSHDOWN_INEXACT;
    else if (can_push_record_filter(f, filters[i])) out[i] = BAMSCAN_PUSHDOWN_INEXACT;
    else out[i] = BAMSCAN_PUSHDOWN_UNSUPPORTED;
  }
  return BAMSCAN_OK;
}

bool filter_is_record_pushable(const BamFile& f, const BamScanFilter& flt) { return can_push_record_filter(f, flt); }

static uint32_t block_of_uoff(const BamFile& f, uint64_t uoff) {
  // first block whose [uoff, uoff+isize) contains the offset (empty members skipped)
  size_t lo = 0, hi = f.blocks.size();
  while (lo < hi) { size_t mid = (lo + hi) / 2; if (f.blocks[mid].uoff + f.blocks[mid].isize <= uoff) lo = mid + 1; else hi = mid; }
  return (uint32_t)lo;
}

int make_plan(BamFile* f, const int32_t* projection, int32_t n_projection, const BamScanFilter* filters, int32_t n_filters,
              int32_t target_partitions, int32_t partition_mode, Plan** out) {
  if (!f->header_ok) { set_error("BAM header could not be read: %s", f->path.c_str()); return BAMSCAN_ERR_FORMAT; }
  std::unique_ptr<Plan> plan(new Plan());
  plan->file = f;
  if (n_projection >= 0) {
    plan->has_projection = true;
    for (int i = 0; i < n_projection; i++) {
      if (projection[i] < 0 || projection[i] >= (int32_t)f->fields.size()) { set_error("projection index %d out of range", projection[i]); return BAMSCAN_ERR_INVALID; }
      plan->projection.push_back(projection[i]);
      plan->out_fields.push_back(f->fields[projection[i]]);
    }
  } else {
    plan->out_fields = f->fields;
  }
  if (target_partitions < 1) target_partitions = 1;

  const uint32_t n_blocks = (uint32_t)f->blocks.size();
  const uint32_t first_block = block_of_uoff(*f, f->first_record_uoff);

  if (partition_mode == BAMSCAN_PARTITION_BLOCK_RANGE) {
    // contiguous block ranges balanced by compressed bytes; ownership = block holding a record's first byte
    uint64_t c0 = first_block < n_blocks ? f->blocks[first_block].coff : f->size, c1 = f->size;
    uint32_t b = first_block;
    for (int p = 0; p < target_partitions; p++) {
      uint64_t cut = c0 + (uint64_t)((__int128)(c1 - c0) * (p + 1) / target_partitions);
      uint32_t e = b;
      while (e < n_blocks && f->blocks[e].coff < cut) e++;
      if (p == target_partitions - 1) e = n_blocks;
      Partition part;
      ScanRange r;
      r.block_begin = b; r.block_end = e;
      r.exact_start = (p == 0);
      r.first_uoff = (p == 0) ? f->first_record_uoff : (b < n_blocks ? f->blocks[b].uoff : f->total_inflated);
      r.stop_uoff = e < n_blocks ? f->blocks[e].uoff : ~0ull;
      bool owns = b < e;
      if (f->format == 2 && owns) {
        // SAM: a record is a line; the host sees whether the byte in front of the range is '\n', so every range starts exactly
        // on its first owned line (one that begins in front of the range's end), in the block that holds it
        r.exact_start = true;
        r.first_uoff = sam_record_start_at(*f, r.first_uoff);
        owns = r.first_uoff < std::min<uint64_t>(r.stop_uoff, f->size);
        if (owns) r.block_begin = block_of_uoff(*f, r.first_uoff);
      }
      if (f->format == 3 && owns) {
        // FASTA: a record belongs to the range that holds its '>'.  Whether the range's first byte starts a line depends on the byte in
        // front of it, so the last non-empty member in front of the range is inflated too, and nothing in it is owned (first_uoff)
        r.exact_start = true;
        r.first_uoff = f->blocks[b].uoff;
        for (uint32_t q = b; q > 0; q--) if (f->blocks[q - 1].isize) { r.block_begin = q - 1; break; }
      }
      if (owns) part.ranges.push_back(r);
      part.estimated_bytes = (e > b && b < n_blocks) ? ((e < n_blocks ? f->blocks[e].coff : f->size) - f->blocks[b].coff) : 0;
      plan->partitions.push_back(part);
      b = e;
    }
    *out = plan.release();
    return BAMSCAN_OK;
  }

  // FASTQ, reference rule (bio-format-fastq/src/physical_exec.rs:94-116, 140-175): a BGZF file with a companion `<path>.gzi`
  // is cut into min(target, blocks) runs of whole blocks by block COUNT (num_blocks / n, the first num_blocks % n runs one
  // longer), where blocks = the GZI entries plus the implicit first member; without a GZI the scan is sequential.
  if (f->format == 1 && target_partitions > 1) {
    std::vector<std::pair<uint64_t, uint64_t>> gzi;
    int rc = load_gzi(f->path + ".gzi", &gzi);
    if (rc == BAMSCAN_OK) {
      gzi.insert(gzi.begin(), std::make_pair(0ull, 0ull));
      std::vector<uint32_t> idx(gzi.size());
      for (size_t i = 0; i < gzi.size(); i++) {
        if (gzi[i].first == f->size && gzi[i].second == f->total_inflated) { idx[i] = n_blocks; continue; }   // an entry for the end of the file: an empty run
        size_t lo = 0, hi = n_blocks;
        while (lo < hi) { size_t mid = (lo + hi) / 2; if (f->blocks[mid].coff < gzi[i].first) lo = mid + 1; else hi = mid; }
        if (lo >= n_blocks || f->blocks[lo].coff != gzi[i].first || f->blocks[lo].uoff != gzi[i].second) {
          set_error("%s.gzi: entry %zu (%llu, %llu) does not name a BGZF member of the file", f->path.c_str(), i, (unsigned long long)gzi[i].first, (unsigned long long)gzi[i].second);
          return BAMSCAN_ERR_FORMAT;
        }
        idx[i] = (uint32_t)lo;
      }
      const size_t num_blocks = gzi.size(), num_partitions = std::min<size_t>((size_t)target_partitions, num_blocks);
      size_t cur = 0;
      for (size_t i = 0; i < num_partitions && cur < num_blocks; i++) {
        const size_t next = cur + num_blocks / num_partitions + (i < num_blocks % num_partitions ? 1 : 0);
        const uint32_t b = idx[cur], e = next >= num_blocks ? n_blocks : idx[next];
        Partition part;
        ScanRange r;
        r.block_begin = b; r.block_end = e;
        r.exact_start = (cur == 0);
        r.first_uoff = b < n_blocks ? f->blocks[b].uoff : f->total_inflated;
        r.stop_uoff = e < n_blocks ? f->blocks[e].uoff : ~0ull;
        if (b < e) part.ranges.push_back(r);
        part.estimated_bytes = b < n_blocks ? (e < n_blocks ? f->blocks[e].coff : f->size) - f->blocks[b].coff : 0;
        plan->partitions.push_back(part);
        cur = next;
      }
      *out = plan.release();
      return BAMSCAN_OK;
    }
    if (rc != BAMSCAN_ERR_IO) return rc;   // an unreadable GZI is "no index" (sequential), a corrupt one is an error
  }

  // reference rule: index present -> region partitions (table_provider.rs:1001-1093)
  if (!f->index_path.empty()) {
    bool handled = false;
    int rc = plan_indexed(f, plan.get(), filters, n_filters, target_partitions, &handled);
    if (rc) return rc;
    if (handled) { *out = plan.release(); return BAMSCAN_OK; }
  }
  // sequential full scan, one partition (table_provider.rs:1097-1114); nothing is pushed down
  Partition part;
  ScanRange r;
  r.block_begin = first_block; r.block_end = n_blocks;
  r.exact_start = true; r.first_uoff = f->first_record_uoff;
  if (r.block_begin < r.block_end) part.ranges.push_back(r);
  part.estimated_bytes = f->size;
  plan->partitions.push_back(part);
  *out = plan.release();
  return BAMSCAN_OK;
}

}  // namespace bamscan
