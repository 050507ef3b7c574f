// host_file.cpp -- BGZF ingest on the host: file load into page-locked memory, BSIZE-chain walk, BAM header,
// tag-type inference sample, index discovery and BAI / CSI parse.
//
// Replaces (reference, datafusion/):
//   bio-format-bam/src/storage.rs:161-169        open_local_bam_sync (BGZF reader + read_header)
//   bio-format-bam/src/table_provider.rs:145-202 discover_tags_from_stream (first N records)
//   bio-format-core/src/index_utils.rs:43-76     index discovery
//   noodles-bam bai::fs::read                    BAI parse (SAMv1 5.2)
// The header block(s) and the inference sample are inflated with zlib on the host: this is planning work
// done once per open, exactly where the reference does it (BamTableProvider::new), not the scan path.
#include <zlib.h>

#include <cctype>
#include <cstdio>
#include <cstring>
#include <sys/stat.h>

#include "bamscan_internal.h"
#include "f32_parse.h"

namespace bamscan {

static inline uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
static inline uint16_t rd16(const uint8_t* p) { uint16_t v; memcpy(&v, p, 2); return v; }

// Sequential inflated-stream reader over the in-memory block table (host zlib) -- header + inference only.
struct HostStream {
  const BamFile& f;
  size_t bi = 0;
  std::vector<uint8_t> buf;
  size_t pos = 0;
  uint64_t base_uoff = 0;    // inflated offset of buf[0]
  explicit HostStream(const BamFile& file) : f(file) {}
  bool fill() {
    while (bi < f.blocks.size()) {
      const BgzfBlock& b = f.blocks[bi++];
      if (b.isize == 0) continue;
      std::vector<uint8_t> out(b.isize);
      z_stream s; memset(&s, 0, sizeof s);
      if (inflateInit2(&s, -15) != Z_OK) return false;
      s.next_in = const_cast<Bytef*>(f.data + b.coff + b.cdata_off); s.avail_in = b.csize - b.cdata_off - 8;
      s.next_out = out.data(); s.avail_out = b.isize;
      int rc = inflate(&s, Z_FINISH); inflateEnd(&s);
      if (rc != Z_STREAM_END || s.total_out != b.isize) return false;
      if ((uint32_t)crc32(crc32(0, nullptr, 0), out.data(), b.isize) != b.crc) return false;
      // drop consumed prefix
      if (pos > 0) { base_uoff += pos; buf.erase(buf.begin(), buf.begin() + (long)pos); pos = 0; }
      buf.insert(buf.end(), out.begin(), out.end());
      return true;
    }
    return false;
  }
  bool need(size_t n) { while (buf.size() - pos < n) if (!fill()) return false; return true; }
  const uint8_t* ptr() const { return buf.data() + pos; }
  void skip(size_t n) { pos += n; }
  uint64_t uoff() const { return base_uoff + pos; }
};

static int walk_blocks(BamFile* f) {
  uint64_t off = 0, uoff = 0;
  while (off < f->size) {
    const uint8_t* p = f->data + off;
    if (f->size - off < 18 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) {
      set_error("invalid BGZF block header at offset %llu (not a BGZF/BAM file?)", (unsigned long long)off);
      return BAMSCAN_ERR_FORMAT;
    }
    uint32_t xlen = rd16(p + 10);
    if (f->size - off < 12ull + xlen) { set_error("truncated BGZF header at offset %llu", (unsigned long long)off); return BAMSCAN_ERR_FORMAT; }
    uint32_t x = 0, bsize = 0; bool found = false;
    while (x + 4 <= xlen) {
      const uint8_t* sf = p + 12 + x; uint32_t slen = rd16(sf + 2);
      if (sf[0] == 'B' && sf[1] == 'C' && slen == 2 && x + 6 <= xlen) { bsize = rd16(sf + 4); found = true; }
      x += 4 + slen;
    }
    uint32_t total = bsize + 1;
    if (!found || total < 12 + xlen + 8 || off + total > f->size) {
      set_error("invalid BGZF BSIZE at offset %llu", (unsigned long long)off);
      return BAMSCAN_ERR_FORMAT;
    }
    BgzfBlock b;
    b.coff = off; b.csize = total; b.cdata_off = 12 + xlen;
    b.crc = rd32(p + total - 8); b.isize = rd32(p + total - 4);
    if (b.isize > 65536) { set_error("BGZF ISIZE %u > 65536 at offset %llu", b.isize, (unsigned long long)off); return BAMSCAN_ERR_FORMAT; }
    b.uoff = uoff; uoff += b.isize;
    f->blocks.push_back(b);
    off += total;
  }
  f->total_inflated = uoff;
  return BAMSCAN_OK;
}

static int load_vcf_header(BamFile* f);

// ---- plain SAM ----
// The text body is described as pseudo-blocks with csize == isize and coff == uoff == the file offset, so that planning, chunking
// and the seam evidence of block-range partitions work on it unchanged.
constexpr uint32_t SAM_BLOCK = 65536;

// @SQ SN / LN -> the reference dictionary (the header's order).  false: the header does not parse (an @SQ line without SN or a
// positive LN that fits an i32, or a name given twice).
static bool sam_header_refs(BamFile* f) {
  size_t pos = 0;
  const std::string& t = f->text;
  while (pos < t.size()) {
    size_t nl = t.find('\n', pos);
    std::string line = t.substr(pos, nl == std::string::npos ? std::string::npos : nl - pos);
    pos = nl == std::string::npos ? t.size() : nl + 1;
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.compare(0, 4, "@SQ\t") != 0) continue;
    std::string sn; long long ln = -1; bool has_sn = false;
    size_t s = 3;
    while (s != std::string::npos && s < line.size()) {
      size_t e = line.find('\t', s + 1);
      std::string tok = line.substr(s + 1, e == std::string::npos ? std::string::npos : e - s - 1);
      if (tok.compare(0, 3, "SN:") == 0) { sn = tok.substr(3); has_sn = true; }
      else if (tok.compare(0, 3, "LN:") == 0) {
        const std::string v = tok.substr(3);
        ln = -1;
        if (!v.empty() && v.size() <= 10 && v.find_first_not_of("0123456789") == std::string::npos) ln = std::stoll(v);
      }
      s = e;
    }
    if (!has_sn || sn.empty() || ln < 1 || ln > 2147483647ll) return false;
    for (const auto& n : f->ref_names) if (n == sn) return false;
    f->ref_names.push_back(sn); f->ref_lens.push_back((int32_t)ln);
  }
  return true;
}

int load_sam(BamFile* f) {
  const uint8_t* d = f->data;
  const uint64_t n = f->size;
  if (n >= 2 && d[0] == 0x1f && d[1] == 0x8b) {
    set_error("%s: gzip / BGZF-compressed SAM is not supported (decompress it, or convert it to BAM)", f->path.c_str());
    return BAMSCAN_ERR_UNSUPPORTED;
  }
  // header: the leading lines that start with '@'
  uint64_t p = 0;
  while (p < n && d[p] == '@') { const void* nl = memchr(d + p, '\n', (size_t)(n - p)); p = nl ? (uint64_t)((const uint8_t*)nl - d) + 1 : n; }
  f->text.assign((const char*)d, (size_t)p);
  f->first_record_uoff = p;
  for (uint64_t o = p; o < n; o += SAM_BLOCK) {
    BgzfBlock b;
    b.coff = b.uoff = o; b.csize = b.isize = (uint32_t)std::min<uint64_t>(SAM_BLOCK, n - o); b.cdata_off = 0; b.crc = 0;
    f->blocks.push_back(b);
  }
  f->total_inflated = n;
  // a header that does not parse gives empty metadata and no references, not an error (as for a BAM, table_provider.rs:423-426)
  f->header_ok = sam_header_refs(f);
  if (!f->header_ok) { f->ref_names.clear(); f->ref_lens.clear(); }
  return BAMSCAN_OK;
}

// BamTableProvider's `is_sam`: a path ending in ".sam", any case (the rule the Python writer uses for its refusal too)
bool is_sam_path(const std::string& path) {
  const size_t n = path.size();
  return n >= 4 && path[n - 4] == '.' && (path[n - 3] | 0x20) == 's' && (path[n - 2] | 0x20) == 'a' && (path[n - 1] | 0x20) == 'm';
}

uint64_t sam_record_start_at(const BamFile& f, uint64_t off) {
  if (off <= f.first_record_uoff) return f.first_record_uoff;
  if (off >= f.size) return f.size;
  if (f.data[off - 1] == '\n') return off;
  const void* nl = memchr(f.data + off, '\n', (size_t)(f.size - off));
  return nl ? (uint64_t)((const uint8_t*)nl - f.data) + 1 : f.size;
}

// [+-]digits (signed) or [+]digits -> *x, saturated far outside every SAM range; false when not an integer
static bool sam_int(const char* s, size_t n, bool allow_neg, long long* x) {
  size_t k = 0; bool neg = false;
  if (k < n && (s[k] == '+' || (allow_neg && s[k] == '-'))) { neg = s[k] == '-'; k++; }
  if (k >= n) return false;
  long long v = 0;
  for (; k < n; k++) { if (s[k] < '0' || s[k] > '9') return false; if (v < (1ll << 40)) v = v * 10 + (s[k] - '0'); }
  *x = neg ? -v : v;
  return true;
}

// The BAM type of one SAM aux field "TG:T:value", as the BAM walk below would report it for the record the transcoder writes:
// an `i` value takes the narrowest type (C / S / I when non-negative, c / s / i when negative), so the value decides between
// Int32 (C, S, c, s, i) and UInt32 (I).  The field is checked by the rules of the device size pass (kernels_sam.cuh::aux_bytes);
// false: the field is malformed (the walk stops there, as the BAM walk does; the scan refuses the line).
static bool sam_aux_type(const char* s, size_t n, std::pair<char, int32_t>* v) {
  auto alpha = [](char c) { return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z'); };
  if (n < 5 || s[2] != ':' || s[4] != ':' || !alpha(s[0]) || !(alpha(s[1]) || (s[1] >= '0' && s[1] <= '9'))) return false;
  const char* val = s + 5;
  const size_t vn = n - 5;
  switch (s[3]) {
    case 'A': *v = {'A', HK_Utf8}; return vn == 1 && val[0] >= '!' && val[0] <= '~';
    case 'i': {
      long long x;
      if (!sam_int(val, vn, true, &x) || x < -2147483648ll || x > 4294967295ll) return false;
      *v = x > 65535 ? std::make_pair('I', (int32_t)HK_UInt32) : std::make_pair('i', (int32_t)HK_Int32);
      return true;
    }
    case 'f': { uint32_t b; *v = {'f', HK_Float32}; return f32_parse(val, (uint32_t)vn, &b); }
    case 'Z':
      for (size_t k = 0; k < vn; k++) if (val[k] < ' ' || val[k] > '~') return false;
      *v = {'Z', HK_Utf8}; return true;
    case 'H':
      if (vn & 1) return false;
      for (size_t k = 0; k < vn; k++) if (!isxdigit((unsigned char)val[k])) return false;
      *v = {'H', HK_Utf8}; return true;
    case 'B': {
      if (vn < 1) return false;
      const char st = val[0];
      int32_t kind; long long lo = 0, hi = 0;
      switch (st) { case 'c': kind = HK_ListInt8; lo = -128; hi = 127; break; case 'C': kind = HK_ListUInt8; hi = 255; break;
                    case 's': kind = HK_ListInt16; lo = -32768; hi = 32767; break; case 'S': kind = HK_ListUInt16; hi = 65535; break;
                    case 'i': kind = HK_ListInt32; lo = -2147483648ll; hi = 2147483647ll; break; case 'I': kind = HK_ListUInt32; hi = 4294967295ll; break;
                    case 'f': kind = HK_ListFloat32; break; default: return false; }
      for (size_t k = 1; k < vn;) {
        if (val[k] != ',') return false;
        size_t j = k + 1;
        while (j < vn && val[j] != ',') j++;
        if (st == 'f') { uint32_t b; if (!f32_parse(val + k + 1, (uint32_t)(j - k - 1), &b)) return false; }
        else { long long x; if (!sam_int(val + k + 1, j - k - 1, true, &x) || x < lo || x > hi) return false; }
        k = j;
      }
      *v = {'B', kind};
      return true;
    }
  }
  return false;
}

// infer_tag_types on a SAM: the aux fields of the first sample_size lines of the body
static int infer_tag_types_sam(const BamFile& f, const std::vector<std::string>& tags, int sample_size,
                               std::map<std::string, std::pair<char, int32_t>>* out, bool all) {
  uint64_t p = f.first_record_uoff;
  for (int count = 0; count < sample_size && p < f.size; count++) {
    const uint8_t* nl = (const uint8_t*)memchr(f.data + p, '\n', (size_t)(f.size - p));
    uint64_t e = nl ? (uint64_t)(nl - f.data) : f.size;
    const uint64_t next = nl ? e + 1 : f.size;
    if (e > p && f.data[e - 1] == '\r') e--;
    const char* line = (const char*)f.data + p;
    const size_t n = (size_t)(e - p);
    p = next;
    size_t k = 0;
    int tabs = 0;
    while (k < n && tabs < 11) { if (line[k] == '\t') tabs++; k++; }
    if (tabs < 11) continue;
    std::map<std::string, std::pair<char, int32_t>> seen;
    while (k < n) {
      size_t j = k;
      while (j < n && line[j] != '\t') j++;
      std::pair<char, int32_t> v;
      if (!sam_aux_type(line + k, j - k, &v)) break;
      std::string tag(line + k, 2);
      if (!seen.count(tag)) seen[tag] = v;
      if (all && !out->count(tag)) (*out)[tag] = v;
      k = j + 1;
    }
    for (const auto& t : tags) {
      if (out->count(t) || t.size() != 2) continue;
      auto it = seen.find(t);
      if (it != seen.end()) (*out)[t] = it->second;
    }
  }
  return BAMSCAN_OK;
}

// ---- VCF header ----
// One ##INFO=<...> or ##FORMAT=<...> line (prefix: the bytes in front of the first key) -> *out.  Values may be quoted ("..." with
// \" and \\ escapes), so a quoted Description may hold ',' '=' '>'.  Keys other than ID, Number, Type and Description are skipped.
// false: the line does not parse (or lacks ID, Number or Type).
static bool vcf_info_line(const std::string& line, size_t prefix, BamFile::VcfInfo* out) {
  size_t k = prefix;
  bool has_id = false, has_num = false, has_type = false;
  for (;;) {
    const size_t eq = line.find('=', k);
    if (eq == std::string::npos) return false;
    const std::string key = line.substr(k, eq - k);
    std::string val;
    k = eq + 1;
    if (k < line.size() && line[k] == '"') {
      for (k++; k < line.size() && line[k] != '"'; k++) {
        if (line[k] == '\\' && k + 1 < line.size()) k++;
        val += line[k];
      }
      if (k >= line.size()) return false;
      k++;
    } else {
      while (k < line.size() && line[k] != ',' && line[k] != '>') val += line[k++];
    }
    if (key == "ID") { out->id = val; has_id = true; }
    else if (key == "Number") { out->number = val; has_num = true; }
    else if (key == "Type") { out->type = val; has_type = true; }
    else if (key == "Description") out->description = val;
    if (k >= line.size()) return false;
    if (line[k] == '>') return has_id && has_num && has_type && !out->id.empty() && k + 1 == line.size();
    if (line[k] != ',') return false;
    k++;
  }
}

// The header of a BGZF VCF: the leading lines up to and including the #CHROM line (host zlib, as for a BAM header).  The first
// line must start with "##fileformat=VCF"; ##INFO lines are kept in header order; the records start behind the #CHROM line.
static int load_vcf_header(BamFile* f) {
  HostStream hs(*f);
  static const char kChrom[] = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO";
  for (uint64_t line_no = 0;; line_no++) {
    size_t nl;
    for (;;) {
      const uint8_t* p = hs.buf.data() + hs.pos;
      const void* q = memchr(p, '\n', hs.buf.size() - hs.pos);
      if (q) { nl = (size_t)((const uint8_t*)q - p); break; }
      if (!hs.fill()) { nl = hs.buf.size() - hs.pos; break; }
    }
    if (nl == 0 && hs.pos >= hs.buf.size()) { set_error("%s: VCF header without a #CHROM line", f->path.c_str()); return BAMSCAN_ERR_FORMAT; }
    std::string line((const char*)hs.ptr(), nl);
    hs.skip(std::min(nl + 1, hs.buf.size() - hs.pos));
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line_no == 0 && line.compare(0, 16, "##fileformat=VCF") != 0) { set_error("%s: not a VCF file (the first line is not ##fileformat=VCF...)", f->path.c_str()); return BAMSCAN_ERR_FORMAT; }
    f->text += line; f->text += '\n';
    if (line.compare(0, 2, "##") == 0) {
      if (line.compare(0, 10, "##FORMAT=<") == 0 && !f->format_fields.empty()) {
        BamFile::VcfInfo fmt;
        if (!vcf_info_line(line, 10, &fmt)) { set_error("%s: malformed ##FORMAT header line: %s", f->path.c_str(), line.c_str()); return BAMSCAN_ERR_FORMAT; }
        for (const auto& o : f->vcf_format)
          if (o.id == fmt.id) { set_error("%s: FORMAT field '%s' is declared twice in the header", f->path.c_str(), fmt.id.c_str()); return BAMSCAN_ERR_FORMAT; }
        f->vcf_format.push_back(fmt);
        continue;
      }
      if (line.compare(0, 8, "##INFO=<") != 0) continue;
      BamFile::VcfInfo info;
      if (!vcf_info_line(line, 8, &info)) { set_error("%s: malformed ##INFO header line: %s", f->path.c_str(), line.c_str()); return BAMSCAN_ERR_FORMAT; }
      for (const auto& o : f->vcf_info)
        if (o.id == info.id) { set_error("%s: INFO field '%s' is declared twice in the header", f->path.c_str(), info.id.c_str()); return BAMSCAN_ERR_FORMAT; }
      f->vcf_info.push_back(info);
      continue;
    }
    const size_t n = sizeof kChrom - 1;
    if (line.compare(0, n, kChrom) != 0 || (line.size() > n && line[n] != '\t')) { set_error("%s: VCF header without a #CHROM line", f->path.c_str()); return BAMSCAN_ERR_FORMAT; }
    if (!f->format_fields.empty() && line.size() > n) {
      // the sample names: the fields behind FORMAT
      std::vector<std::string> extra;
      for (size_t a = n + 1;;) {
        const size_t t = line.find('\t', a);
        extra.push_back(line.substr(a, t == std::string::npos ? std::string::npos : t - a));
        if (t == std::string::npos) break;
        a = t + 1;
      }
      if (extra[0] != "FORMAT") { set_error("%s: the #CHROM line has fields behind INFO but the first one is not FORMAT", f->path.c_str()); return BAMSCAN_ERR_FORMAT; }
      f->vcf_samples.assign(extra.begin() + 1, extra.end());
    }
    f->first_record_uoff = hs.uoff();
    f->header_ok = true;
    return BAMSCAN_OK;
  }
}

void release_file(BamFile* f) {
  if (!f->data) return;
  if (f->mapped) unmap_file_pinned(f->data, f->size, f->registered); else pinned_free(f->data);
  f->data = nullptr;
}

int load_file(BamFile* f) {
  FILE* fp = fopen(f->path.c_str(), "rb");
  if (!fp) { set_error("cannot open %s", f->path.c_str()); return BAMSCAN_ERR_IO; }
  struct stat st;
  if (fstat(fileno(fp), &st) != 0) { fclose(fp); set_error("cannot stat %s", f->path.c_str()); return BAMSCAN_ERR_IO; }
  f->size = (uint64_t)st.st_size;
  if (f->size >= (1u << 20)) {   // large files: read-only mapping (page cache shared between the per-GPU processes of one node)
    f->data = (uint8_t*)map_file_pinned(f->path.c_str(), f->size, &f->registered);
    f->mapped = f->data != nullptr;
    if (!f->data) { fclose(fp); set_error("cannot map %s read-only", f->path.c_str()); return BAMSCAN_ERR_IO; }
  }
  if (!f->data) {                 // small file: a private copy (at most 1 MiB)
    f->data = (uint8_t*)pinned_alloc(f->size + 4096);
    if (!f->data) { fclose(fp); return BAMSCAN_ERR_CUDA; }
    f->pinned = true;
    uint64_t got = 0;
    while (got < f->size) {
      size_t n = fread(f->data + got, 1, (size_t)std::min<uint64_t>(f->size - got, 1ull << 30), fp);
      if (n == 0) break;
      got += n;
    }
    if (got != f->size) { fclose(fp); set_error("short read on %s", f->path.c_str()); return BAMSCAN_ERR_IO; }
    memset(f->data + f->size, 0, 4096);
  }
  fclose(fp);
  if (f->format == FMT_SAM) return load_sam(f);
  int rc = walk_blocks(f);
  if (rc) return rc;
  if (f->format == FMT_FASTQ || f->format == FMT_FASTA) { f->first_record_uoff = 0; f->header_ok = true; return BAMSCAN_OK; }     // FASTQ, FASTA: no header
  if (f->format == FMT_VCF) return load_vcf_header(f);

  // BAM header (noodles-bam read_header): magic, l_text, text, n_ref, (l_name, name, l_ref) * n_ref
  HostStream hs(*f);
  if (!hs.need(12) || memcmp(hs.ptr(), "BAM\1", 4) != 0) { set_error("%s: missing BAM magic", f->path.c_str()); return BAMSCAN_ERR_FORMAT; }
  uint32_t l_text = rd32(hs.ptr() + 4); hs.skip(8);
  if (!hs.need((size_t)l_text + 4)) { set_error("truncated BAM header text"); return BAMSCAN_ERR_FORMAT; }
  f->text.assign((const char*)hs.ptr(), l_text);
  while (!f->text.empty() && f->text.back() == '\0') f->text.pop_back();
  hs.skip(l_text);
  uint32_t n_ref = rd32(hs.ptr()); hs.skip(4);
  for (uint32_t i = 0; i < n_ref; i++) {
    if (!hs.need(4)) { set_error("truncated BAM reference list"); return BAMSCAN_ERR_FORMAT; }
    uint32_t l_name = rd32(hs.ptr()); hs.skip(4);
    if (!hs.need((size_t)l_name + 4)) { set_error("truncated BAM reference list"); return BAMSCAN_ERR_FORMAT; }
    std::string name((const char*)hs.ptr(), l_name);
    while (!name.empty() && name.back() == '\0') name.pop_back();
    hs.skip(l_name);
    f->ref_names.push_back(name);
    f->ref_lens.push_back((int32_t)rd32(hs.ptr())); hs.skip(4);
  }
  f->first_record_uoff = hs.uoff();
  f->header_ok = true;
  return BAMSCAN_OK;
}

// table_provider.rs:145-202 + tag_registry.rs:772-792
// `all` (BamTableProvider::describe, table_provider.rs:715-745): every tag met in the sample, first occurrence wins.
int infer_tag_types(const BamFile& f, const std::vector<std::string>& tags, int sample_size,
                    std::map<std::string, std::pair<char, int32_t>>* out, bool all) {
  if (f.format == FMT_SAM) return infer_tag_types_sam(f, tags, sample_size, out, all);
  HostStream hs(f);
  // position on the first record
  while (hs.base_uoff + hs.buf.size() <= f.first_record_uoff) if (!hs.fill()) return BAMSCAN_OK;
  hs.pos = (size_t)(f.first_record_uoff - hs.base_uoff);
  for (int count = 0; count < sample_size; count++) {
    if (!hs.need(4)) break;
    uint32_t bs = rd32(hs.ptr());
    if (bs < 32 || !hs.need(4 + (size_t)bs)) break;
    const uint8_t* rec = hs.ptr() + 4;
    uint32_t l_name = rec[8], n_cig = rd16(rec + 12), l_seq = rd32(rec + 16);
    size_t a = 32 + (size_t)l_name + 4 * (size_t)n_cig + ((size_t)l_seq + 1) / 2 + l_seq;
    std::map<std::string, std::pair<char, int32_t>> seen;   // Data::get returns the first field with the tag
    while (a + 3 <= bs) {
      std::string tag((const char*)rec + a, 2); char ty = (char)rec[a + 2]; a += 3;
      size_t sz;
      std::pair<char, int32_t> v;
      if (ty == 'A') { sz = 1; v = {'A', HK_Utf8}; }
      else if (ty == 'c' || ty == 'C') { sz = 1; v = {'i', HK_Int32}; }
      else if (ty == 's' || ty == 'S') { sz = 2; v = {'i', HK_Int32}; }
      else if (ty == 'i') { sz = 4; v = {'i', HK_Int32}; }
      else if (ty == 'I') { sz = 4; v = {'I', HK_UInt32}; }
      else if (ty == 'f') { sz = 4; v = {'f', HK_Float32}; }
      else if (ty == 'Z' || ty == 'H') { const void* z = memchr(rec + a, 0, bs - a); if (!z) break; sz = (size_t)((const uint8_t*)z - (rec + a)) + 1; v = {ty, HK_Utf8}; }
      else if (ty == 'B') {
        if (a + 5 > bs) break;
        char st = (char)rec[a]; uint32_t cnt = rd32(rec + a + 1);
        int es, kind;
        switch (st) { case 'c': es = 1; kind = HK_ListInt8; break; case 'C': es = 1; kind = HK_ListUInt8; break; case 's': es = 2; kind = HK_ListInt16; break;
                      case 'S': es = 2; kind = HK_ListUInt16; break; case 'i': es = 4; kind = HK_ListInt32; break; case 'I': es = 4; kind = HK_ListUInt32; break;
                      case 'f': es = 4; kind = HK_ListFloat32; break; default: es = 0; kind = 0; }
        if (!es) break;
        sz = 5 + (size_t)cnt * es; v = {'B', kind};
      } else break;
      if (a + sz > bs) break;
      if (!seen.count(tag)) seen[tag] = v;
      if (all && !out->count(tag)) (*out)[tag] = v;
      a += sz;
    }
    for (const auto& t : tags) {
      if (out->count(t) || t.size() != 2) continue;
      auto it = seen.find(t);
      if (it != seen.end()) (*out)[t] = it->second;
    }
    hs.skip(4 + (size_t)bs);
  }
  return BAMSCAN_OK;
}

static bool file_exists(const std::string& p) { struct stat st; return stat(p.c_str(), &st) == 0 && S_ISREG(st.st_mode); }

// index_utils.rs:43-76: <path>.bai, <stem>.bai, then <path>.csi
std::string discover_index(const std::string& path) {
  std::string c1 = path + ".bai";
  if (file_exists(c1)) return c1;
  size_t dot = path.find_last_of('.'), slash = path.find_last_of('/');
  if (dot != std::string::npos && (slash == std::string::npos || dot > slash)) {
    std::string c2 = path.substr(0, dot) + ".bai";
    if (file_exists(c2)) return c2;
  }
  std::string c3 = path + ".csi";   // discover_bam_index: BAI first, then CSI (index_utils.rs:68-76)
  if (file_exists(c3)) return c3;
  return std::string();
}

// A CSI file is BGZF: inflate every gzip member (host zlib, planning work) into one buffer.
static bool gunzip_members(const std::vector<uint8_t>& in, std::vector<uint8_t>* out) {
  size_t p = 0;
  while (p < in.size()) {
    z_stream s; memset(&s, 0, sizeof s);
    if (inflateInit2(&s, 15 + 16) != Z_OK) return false;
    s.next_in = const_cast<Bytef*>(in.data() + p); s.avail_in = (uInt)std::min<size_t>(in.size() - p, 1u << 30);
    int rc = Z_OK;
    while (rc == Z_OK) {
      uint8_t tmp[65536]; s.next_out = tmp; s.avail_out = sizeof tmp;
      rc = inflate(&s, Z_NO_FLUSH);
      if (rc != Z_OK && rc != Z_STREAM_END) { inflateEnd(&s); return false; }
      out->insert(out->end(), tmp, tmp + (sizeof tmp - s.avail_out));
      if (out->size() > (1ull << 32)) { inflateEnd(&s); return false; }   // an index of more than 4 GiB is not an index
    }
    p += s.total_in; inflateEnd(&s);
  }
  return true;
}

// CSIv1 (SAM/BAM specification group, "Coordinate Sorted Index"): magic, min_shift, depth, l_aux, aux, n_ref,
// per reference n_bin x { bin, loffset, n_chunk, chunks }, optional n_no_coor.  noodles-csi reads the same layout; the reference
// discovers `<path>.csi` (index_utils.rs:54-56, 68-76) and then hands it to `bam::bai::fs::read`, which refuses the magic, so an
// indexed scan over a CSI is an error there; this build reads it (same planner, bin scheme from the file).
static int parse_csi(const std::string& path, const std::vector<uint8_t>& d, BaiIndex* out) {
  size_t p = 0;
  auto need = [&](uint64_t k) { return k <= d.size() - p; };
  if (d.size() < 16 || memcmp(d.data(), "CSI\1", 4) != 0) { set_error("%s: missing CSI magic", path.c_str()); return BAMSCAN_ERR_FORMAT; }
  const int32_t min_shift = (int32_t)rd32(d.data() + 4), depth = (int32_t)rd32(d.data() + 8);
  const uint32_t l_aux = rd32(d.data() + 12); p = 16;
  // bin ids are 32-bit: first_bin(depth + 1) + 1 must fit => depth <= 9; positions stay below 2^44 here
  if (min_shift < 1 || depth < 1 || depth > 9 || min_shift + 3 * depth > 44) { set_error("%s: CSI min_shift %d / depth %d not supported", path.c_str(), min_shift, depth); return BAMSCAN_ERR_UNSUPPORTED; }
  out->csi = true; out->min_shift = min_shift; out->depth = depth;
  if (!need((uint64_t)l_aux + 4)) goto trunc;
  p += l_aux;
  {
    const uint32_t n_ref = rd32(d.data() + p); p += 4;
    if ((uint64_t)n_ref * 4ull > d.size() - p) { set_error("%s: CSI n_ref %u exceeds the file size", path.c_str(), n_ref); return BAMSCAN_ERR_FORMAT; }
    const uint32_t meta = out->meta_bin();
    out->refs.resize(n_ref);
    for (uint32_t r = 0; r < n_ref; r++) {
      if (!need(4)) goto trunc;
      const uint32_t n_bin = rd32(d.data() + p); p += 4;
      BaiRef& R = out->refs[r];
      for (uint32_t b = 0; b < n_bin; b++) {
        if (!need(16)) goto trunc;
        const uint32_t bin = rd32(d.data() + p); uint64_t loff; memcpy(&loff, d.data() + p + 4, 8);
        const uint32_t n_chunk = rd32(d.data() + p + 12); p += 16;
        if (!need(16ull * n_chunk)) goto trunc;
        if (bin == meta && n_chunk == 2) {
          R.has_meta = true;
          memcpy(&R.meta_beg, d.data() + p, 8); memcpy(&R.meta_end, d.data() + p + 8, 8);
          memcpy(&R.n_mapped, d.data() + p + 16, 8); memcpy(&R.n_unmapped, d.data() + p + 24, 8);
        } else {
          auto& v = R.bins[bin];
          for (uint32_t c = 0; c < n_chunk; c++) { BaiChunk ch; memcpy(&ch.beg, d.data() + p + 16 * c, 8); memcpy(&ch.end, d.data() + p + 16 * c + 8, 8); v.push_back(ch); }
          R.loffset[bin] = loff;
        }
        p += 16ull * n_chunk;
      }
    }
    if (need(8)) { memcpy(&out->n_no_coor, d.data() + p, 8); out->has_no_coor = true; }
  }
  return BAMSCAN_OK;
trunc:
  set_error("%s: truncated CSI", path.c_str());
  return BAMSCAN_ERR_FORMAT;
}

// GZI (bgzip -i; noodles-bgzf gzi::fs::read): u64 count, then count x (compressed offset, inflated offset), little endian.
int load_gzi(const std::string& path, std::vector<std::pair<uint64_t, uint64_t>>* out) {
  FILE* fp = fopen(path.c_str(), "rb");
  if (!fp) return BAMSCAN_ERR_IO;
  std::vector<uint8_t> d;
  uint8_t tmp[65536]; size_t n;
  while ((n = fread(tmp, 1, sizeof tmp, fp)) > 0) d.insert(d.end(), tmp, tmp + n);
  fclose(fp);
  uint64_t cnt = 0;
  if (d.size() >= 8) memcpy(&cnt, d.data(), 8);
  if (d.size() < 8 || cnt > (d.size() - 8) / 16 || d.size() != 8 + 16 * cnt) { set_error("%s: not a GZI index (size %zu, count %llu)", path.c_str(), d.size(), (unsigned long long)cnt); return BAMSCAN_ERR_FORMAT; }
  out->resize((size_t)cnt);
  for (uint64_t i = 0; i < cnt; i++) { memcpy(&(*out)[i].first, d.data() + 8 + 16 * i, 8); memcpy(&(*out)[i].second, d.data() + 16 + 16 * i, 8); }
  for (uint64_t i = 1; i < cnt; i++)
    if ((*out)[i].first <= (*out)[i - 1].first) { set_error("%s: GZI offsets are not increasing", path.c_str()); return BAMSCAN_ERR_FORMAT; }
  return BAMSCAN_OK;
}

int load_bai(const std::string& path, BaiIndex* out) {
  FILE* fp = fopen(path.c_str(), "rb");
  if (!fp) { set_error("cannot open index %s", path.c_str()); return BAMSCAN_ERR_IO; }
  std::vector<uint8_t> d;
  uint8_t tmp[65536]; size_t n;
  while ((n = fread(tmp, 1, sizeof tmp, fp)) > 0) d.insert(d.end(), tmp, tmp + n);
  fclose(fp);
  if (d.size() >= 4 && d[0] == 0x1f && d[1] == 0x8b) {   // BGZF container: a CSI
    std::vector<uint8_t> u;
    if (!gunzip_members(d, &u)) { set_error("%s: cannot inflate the index", path.c_str()); return BAMSCAN_ERR_FORMAT; }
    return parse_csi(path, u, out);
  }
  if (d.size() >= 4 && memcmp(d.data(), "CSI\1", 4) == 0) return parse_csi(path, d, out);
  size_t p = 0;
  auto need = [&](size_t k) { return p + k <= d.size(); };
  if (!need(8) || memcmp(d.data(), "BAI\1", 4) != 0) { set_error("%s: missing BAI magic", path.c_str()); return BAMSCAN_ERR_FORMAT; }
  uint32_t n_ref = rd32(d.data() + 4); p = 8;
  // every reference takes at least 8 bytes (n_bin, n_intv): a count the file cannot hold is a corrupt index, not an allocation
  if ((uint64_t)n_ref * 8ull > d.size() - p) { set_error("%s: BAI n_ref %u exceeds the file size", path.c_str(), n_ref); return BAMSCAN_ERR_FORMAT; }
  out->refs.resize(n_ref);
  for (uint32_t r = 0; r < n_ref; r++) {
    if (!need(4)) goto trunc;
    {
      uint32_t n_bin = rd32(d.data() + p); p += 4;
      for (uint32_t b = 0; b < n_bin; b++) {
        if (!need(8)) goto trunc;
        uint32_t bin = rd32(d.data() + p), n_chunk = rd32(d.data() + p + 4); p += 8;
        if (!need(16ull * n_chunk)) goto trunc;
        if (bin == 37450 && n_chunk == 2) {
          BaiRef& R = out->refs[r]; R.has_meta = true;
          memcpy(&R.meta_beg, d.data() + p, 8); memcpy(&R.meta_end, d.data() + p + 8, 8);
          memcpy(&R.n_mapped, d.data() + p + 16, 8); memcpy(&R.n_unmapped, d.data() + p + 24, 8);
        } else {
          auto& v = out->refs[r].bins[bin];
          for (uint32_t c = 0; c < n_chunk; c++) { BaiChunk ch; memcpy(&ch.beg, d.data() + p + 16 * c, 8); memcpy(&ch.end, d.data() + p + 16 * c + 8, 8); v.push_back(ch); }
        }
        p += 16ull * n_chunk;
      }
      if (!need(4)) goto trunc;
      uint32_t n_intv = rd32(d.data() + p); p += 4;
      if (!need(8ull * n_intv)) goto trunc;
      out->refs[r].intervals.resize(n_intv);
      if (n_intv) memcpy(out->refs[r].intervals.data(), d.data() + p, 8ull * n_intv);
      p += 8ull * n_intv;
    }
  }
  if (need(8)) { memcpy(&out->n_no_coor, d.data() + p, 8); out->has_no_coor = true; }
  return BAMSCAN_OK;
trunc:
  set_error("%s: truncated BAI", path.c_str());
  return BAMSCAN_ERR_FORMAT;
}

}  // namespace bamscan
