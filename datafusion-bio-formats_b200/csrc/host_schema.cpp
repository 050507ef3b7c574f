// host_schema.cpp -- Arrow schema of the BAM table: 12 core columns + typed tag columns + bio.bam.* metadata.
//
// Replaces (reference, datafusion/):
//   bio-format-bam/src/table_provider.rs:42-140   determine_schema (inferred > hints > registry > Utf8)
//   bio-format-core/src/tag_registry.rs:131-792   registry, hint grammar, type formatting
//   bio-format-core/src/metadata.rs:321-485       extract_header_metadata (SAM header -> JSON strings)
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "bamscan_internal.h"

namespace bamscan {

static thread_local char g_err[1024];
void set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}
const char* last_error_cstr() { return g_err; }

const std::map<std::string, TagDef>& known_tags() {
  static const std::map<std::string, TagDef> tags = [] {
    std::map<std::string, TagDef> m;
    enum { K_Int32 = HK_Int32, K_Utf8 = HK_Utf8, K_ListUInt8 = HK_ListUInt8, K_ListUInt16 = HK_ListUInt16, K_ListUInt32 = HK_ListUInt32 };
#define TAGDEF(tag, sam, kind, desc) m[tag] = TagDef{tag, sam, kind, desc};
#include "tag_registry_data.inc"
#undef TAGDEF
    return m;
  }();
  return tags;
}

static int32_t subtype_kind(char st) {
  switch (st) { case 'c': return HK_ListInt8; case 'C': return HK_ListUInt8; case 's': return HK_ListInt16; case 'S': return HK_ListUInt16;
                case 'i': return HK_ListInt32; case 'I': return HK_ListUInt32; case 'f': return HK_ListFloat32; }
  return 0;
}
static char kind_subtype(int32_t kind) {
  switch (kind) { case HK_ListInt8: return 'c'; case HK_ListUInt8: return 'C'; case HK_ListInt16: return 's'; case HK_ListUInt16: return 'S';
                  case HK_ListInt32: return 'i'; case HK_ListUInt32: return 'I'; case HK_ListFloat32: return 'f'; }
  return 0;
}

std::string format_sam_tag_type(char sam_type, int32_t kind) {
  if (sam_type == 'B' && kind_subtype(kind)) return std::string("B:") + kind_subtype(kind);
  return std::string(1, sam_type);
}

bool parse_tag_type_hints(const std::vector<std::string>& hints, std::map<std::string, std::pair<char, int32_t>>* out) {
  for (const std::string& hint : hints) {
    std::vector<std::string> parts;
    size_t s = 0;
    for (;;) { size_t c = hint.find(':', s); parts.push_back(hint.substr(s, c == std::string::npos ? c : c - s)); if (c == std::string::npos) break; s = c + 1; }
    if (parts.size() == 2) {
      if (parts[1].size() != 1) { set_error("Invalid tag type hint '%s': TYPE must be a single character", hint.c_str()); return false; }
      char t = parts[1][0];
      if (t == 'B') { set_error("Invalid tag type hint '%s': array type 'B' requires a subtype. Use 'TAG:B:c|C|s|S|i|I|f'", hint.c_str()); return false; }
      int32_t kind;
      switch (t) {
        case 'A': case 'Z': case 'H': kind = HK_Utf8; break;
        case 'c': case 's': case 'i': kind = HK_Int32; break;
        case 'C': case 'S': case 'I': kind = HK_UInt32; break;
        case 'f': kind = HK_Float32; break;
        default: set_error("Invalid tag type hint '%s': unsupported SAM type '%c'. Supported types: A, c, C, s, S, i, I, f, Z, H", hint.c_str(), t); return false;
      }
      (*out)[parts[0]] = {t, kind};
    } else if (parts.size() == 3 && parts[1] == "B") {
      if (parts[2].size() != 1) { set_error("Invalid tag type hint '%s': array subtype must be a single character", hint.c_str()); return false; }
      int32_t kind = subtype_kind(parts[2][0]);
      if (!kind) { set_error("Invalid tag type hint '%s': unsupported array subtype '%c'. Supported subtypes: c, C, s, S, i, I, f", hint.c_str(), parts[2][0]); return false; }
      (*out)[parts[0]] = {'B', kind};
    } else {
      set_error("Invalid tag type hint '%s': expected 'TAG:TYPE' or 'TAG:B:SUBTYPE' format", hint.c_str());
      return false;
    }
  }
  return true;
}

// ---------------------------------------------------------------------------------------------
// SAM header text -> bio.bam.* metadata (metadata.rs:321-485)
static std::string json_escape(const std::string& s) {
  std::string o = "\"";
  for (unsigned char c : s) {
    switch (c) {
      case '"': o += "\\\""; break;
      case '\\': o += "\\\\"; break;
      case '\n': o += "\\n"; break;
      case '\r': o += "\\r"; break;
      case '\t': o += "\\t"; break;
      case '\b': o += "\\b"; break;
      case '\f': o += "\\f"; break;
      default:
        if (c < 0x20) { char t[8]; snprintf(t, sizeof t, "\\u%04x", c); o += t; }
        else o += (char)c;
    }
  }
  return o + "\"";
}

typedef std::vector<std::pair<std::string, std::string>> KV;
static const std::string* kv_get(const KV& kv, const char* k) { for (auto& p : kv) if (p.first == k) return &p.second; return nullptr; }

static std::string other_fields_json(const KV& kv, std::initializer_list<const char*> skip) {
  std::string o; bool first = true;
  for (auto& p : kv) {
    bool sk = false;
    for (const char* s : skip) if (p.first == s) sk = true;
    if (sk) continue;
    o += first ? "" : ","; first = false;
    o += json_escape(p.first) + ":" + json_escape(p.second);
  }
  return o;
}

static void header_metadata(BamFile* f) {
  KV& md = f->schema_metadata;
  std::string sq, rg, pg, co;
  size_t pos = 0;
  const std::string& text = f->text;
  while (pos < text.size()) {
    size_t nl = text.find('\n', pos);
    std::string line = text.substr(pos, nl == std::string::npos ? std::string::npos : nl - pos);
    pos = nl == std::string::npos ? text.size() : nl + 1;
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.size() < 3 || line[0] != '@') continue;
    std::string kind = line.substr(0, 3);
    if (kind == "@CO") { co += (co.empty() ? "" : ",") + json_escape(line.size() > 4 ? line.substr(4) : std::string()); continue; }
    KV kv;
    size_t s = line.find('\t');
    while (s != std::string::npos) {
      size_t e = line.find('\t', s + 1);
      std::string tok = line.substr(s + 1, e == std::string::npos ? std::string::npos : e - s - 1);
      if (tok.size() >= 3 && tok[2] == ':') {
        bool dup = false;
        for (auto& p : kv) if (p.first == tok.substr(0, 2)) { p.second = tok.substr(3); dup = true; }
        if (!dup) kv.push_back({tok.substr(0, 2), tok.substr(3)});
      }
      s = e;
    }
    if (kind == "@HD") {
      if (auto v = kv_get(kv, "VN")) md.push_back({"bio.bam.file_format_version", *v});
      if (auto v = kv_get(kv, "SO")) md.push_back({"bio.bam.sort_order", *v});
      if (auto v = kv_get(kv, "GO")) md.push_back({"bio.bam.group_order", *v});
      if (auto v = kv_get(kv, "SS")) md.push_back({"bio.bam.subsort_order", *v});
    } else if (kind == "@SQ") {
      const std::string* sn = kv_get(kv, "SN"); const std::string* ln = kv_get(kv, "LN");
      std::string name = sn ? *sn : std::string();
      uint64_t len = ln ? strtoull(ln->c_str(), nullptr, 10) : 0;
      f->meta_ref_names.push_back(name); f->meta_ref_lens.push_back(len);
      std::string o = "{\"name\":" + json_escape(name) + ",\"length\":" + std::to_string(len);
      std::string other = other_fields_json(kv, {"SN", "LN"});
      if (!other.empty()) o += ",\"other_fields\":{" + other + "}";
      sq += (sq.empty() ? "" : ",") + o + "}";
    } else if (kind == "@RG") {
      const std::string* id = kv_get(kv, "ID");
      std::string o = "{\"id\":" + json_escape(id ? *id : std::string());
      static const char* keys[4][2] = {{"sample", "SM"}, {"platform", "PL"}, {"library", "LB"}, {"description", "DS"}};
      for (auto& k : keys) if (auto v = kv_get(kv, k[1])) o += std::string(",\"") + k[0] + "\":" + json_escape(*v);
      std::string other = other_fields_json(kv, {"ID", "SM", "PL", "LB", "DS"});
      if (!other.empty()) o += ",\"other_fields\":{" + other + "}";
      rg += (rg.empty() ? "" : ",") + o + "}";
    } else if (kind == "@PG") {
      const std::string* id = kv_get(kv, "ID");
      std::string o = "{\"id\":" + json_escape(id ? *id : std::string());
      static const char* keys[3][2] = {{"name", "PN"}, {"version", "VN"}, {"command_line", "CL"}};
      for (auto& k : keys) if (auto v = kv_get(kv, k[1])) o += std::string(",\"") + k[0] + "\":" + json_escape(*v);
      std::string other = other_fields_json(kv, {"ID", "PN", "VN", "CL"});
      if (!other.empty()) o += ",\"other_fields\":{" + other + "}";
      pg += (pg.empty() ? "" : ",") + o + "}";
    }
  }
  if (!sq.empty()) md.push_back({"bio.bam.reference_sequences", "[" + sq + "]"});
  if (!rg.empty()) md.push_back({"bio.bam.read_groups", "[" + rg + "]"});
  if (!pg.empty()) md.push_back({"bio.bam.program_info", "[" + pg + "]"});
  if (!co.empty()) md.push_back({"bio.bam.comments", "[" + co + "]"});
}

int build_schema(BamFile* f, const BamScanOptions* opt) {
  std::map<std::string, std::pair<char, int32_t>> hints, inferred;
  bool has_hints = opt->n_tag_type_hints > 0 && opt->tag_type_hints;
  if (has_hints) {
    std::vector<std::string> hv;
    for (int i = 0; i < opt->n_tag_type_hints; i++) hv.push_back(opt->tag_type_hints[i]);
    if (!parse_tag_type_hints(hv, &hints)) return BAMSCAN_ERR_INVALID;
  }
  if (f->header_ok) header_metadata(f);
  const auto& reg = known_tags();
  bool did_infer = false;
  if (opt->infer_tag_types && f->has_tag_fields && f->header_ok) {
    std::vector<std::string> unknown;
    for (auto& t : f->tag_fields) if (!reg.count(t)) unknown.push_back(t);
    if (!unknown.empty()) { infer_tag_types(*f, unknown, opt->infer_tag_sample_size, &inferred); did_infer = true; }
  }
  f->fields = {
      {"name", HK_Utf8, true, {}}, {"chrom", HK_Utf8, true, {}}, {"start", HK_UInt32, true, {}}, {"end", HK_UInt32, true, {}},
      {"flags", HK_UInt32, false, {}}, {"cigar", f->binary_cigar ? HK_Binary : HK_Utf8, false, {}}, {"mapping_quality", HK_UInt32, false, {}},
      {"mate_chrom", HK_Utf8, true, {}}, {"mate_start", HK_UInt32, true, {}}, {"sequence", HK_Utf8, false, {}},
      {"quality_scores", HK_Utf8, false, {}}, {"template_length", HK_Int32, false, {}}};
  if (f->has_tag_fields) {
    for (auto& tag : f->tag_fields) {
      char sam; int32_t kind; std::string desc;
      auto r = reg.find(tag);
      if (did_infer && inferred.count(tag)) {
        sam = inferred[tag].first; kind = inferred[tag].second;
        desc = r != reg.end() ? r->second.description : std::string("Tag type discovered from file (") + sam + ")";
      } else if (has_hints && hints.count(tag)) {
        sam = hints[tag].first; kind = hints[tag].second;
        desc = r != reg.end() ? r->second.description : std::string("Tag type from user hint (") + sam + ")";
      } else if (r != reg.end()) { sam = r->second.sam_type; kind = r->second.kind; desc = r->second.description; }
      else { sam = 'Z'; kind = HK_Utf8; desc = "Unknown tag"; }
      FieldDef fd{tag, kind, true, {}};
      fd.metadata.push_back({"bio.bam.tag.tag", tag});
      fd.metadata.push_back({"bio.bam.tag.type", format_sam_tag_type(sam, kind)});
      fd.metadata.push_back({"bio.bam.tag.description", desc});
      f->fields.push_back(fd);
    }
  }
  f->schema_metadata.push_back({"bio.coordinate_system_zero_based", f->zero_based ? "true" : "false"});
  if (f->binary_cigar) f->schema_metadata.push_back({"bio.bam.binary_cigar", "true"});
  return BAMSCAN_OK;
}

// VCF: chrom, start, end, id, ref, alt, qual, filter, then one column per selected ##INFO field (DESIGN 3.11).  Type=Flag ->
// Boolean (not null); Number=1 -> Int32 / Float32 / Utf8; any other Number -> a list of those.  The field metadata carries the
// header's Number, Type and Description.  BAMSCAN_ERR_SCHEMA names the field: an ID the header does not declare, an ID equal to a
// fixed column's name, an unknown Type, Number=0 on a type other than Flag.
int build_vcf_schema(BamFile* f, const BamScanOptions* opt) {
  static const char* fixed[] = {"chrom", "start", "end", "id", "ref", "alt", "qual", "filter"};
  f->fields = {{"chrom", HK_Utf8, false, {}}, {"start", HK_UInt32, false, {}}, {"end", HK_UInt32, false, {}}, {"id", HK_Utf8, true, {}},
               {"ref", HK_Utf8, false, {}}, {"alt", HK_Utf8, true, {}}, {"qual", HK_Float32, true, {}}, {"filter", HK_Utf8, true, {}}};
  std::vector<const BamFile::VcfInfo*> sel;
  if (opt->has_tag_fields) {
    for (int i = 0; i < opt->n_tag_fields && opt->tag_fields; i++) {
      const std::string id = opt->tag_fields[i] ? opt->tag_fields[i] : "";
      const BamFile::VcfInfo* hit = nullptr;
      for (const auto& d : f->vcf_info) if (d.id == id) { hit = &d; break; }
      if (!hit) { set_error("INFO field '%s' is not declared in the VCF header", id.c_str()); return BAMSCAN_ERR_SCHEMA; }
      if (std::find(sel.begin(), sel.end(), hit) != sel.end()) { set_error("INFO field '%s' is selected twice", id.c_str()); return BAMSCAN_ERR_SCHEMA; }
      sel.push_back(hit);
    }
  } else {
    for (const auto& d : f->vcf_info) sel.push_back(&d);
  }
  for (const BamFile::VcfInfo* d : sel) {
    for (const char* c : fixed)
      if (d->id == c) { set_error("INFO field '%s' has the name of a fixed VCF column", d->id.c_str()); return BAMSCAN_ERR_SCHEMA; }
    int32_t scalar;
    if (d->type == "Flag") scalar = HK_Boolean;
    else if (d->type == "Integer") scalar = HK_Int32;
    else if (d->type == "Float") scalar = HK_Float32;
    else if (d->type == "String" || d->type == "Character") scalar = HK_Utf8;
    else { set_error("INFO field '%s' has the unknown Type '%s'", d->id.c_str(), d->type.c_str()); return BAMSCAN_ERR_SCHEMA; }
    if (scalar != HK_Boolean && d->number == "0") { set_error("INFO field '%s' has Number=0 but Type=%s (only a Flag may have Number=0)", d->id.c_str(), d->type.c_str()); return BAMSCAN_ERR_SCHEMA; }
    int32_t kind = scalar;
    if (scalar != HK_Boolean && d->number != "1") kind = scalar == HK_Int32 ? HK_ListInt32 : scalar == HK_Float32 ? HK_ListFloat32 : HK_ListUtf8;
    FieldDef fd{d->id, kind, scalar != HK_Boolean, {}};
    fd.metadata = {{"bio.vcf.info.number", d->number}, {"bio.vcf.info.type", d->type}, {"bio.vcf.info.description", d->description}};
    f->fields.push_back(fd);
  }
  f->vcf_info_end = (int32_t)f->fields.size();
  // FORMAT columns (format_fields; none when empty): format_<ID>, one element per sample
  const std::vector<std::string>& ff = f->format_fields;
  if (ff.empty()) return BAMSCAN_OK;
  if (ff.size() > 16) { set_error("more than 16 FORMAT fields (%zu) are not supported by this build", ff.size()); return BAMSCAN_ERR_UNSUPPORTED; }
  if (f->vcf_samples.empty()) { set_error("FORMAT field '%s' is selected but the VCF header has no samples", ff[0].c_str()); return BAMSCAN_ERR_SCHEMA; }
  for (size_t i = 0; i < ff.size(); i++) {
    const BamFile::VcfInfo* d = nullptr;
    for (const auto& x : f->vcf_format) if (x.id == ff[i]) { d = &x; break; }
    if (!d) { set_error("FORMAT field '%s' is not declared in the VCF header", ff[i].c_str()); return BAMSCAN_ERR_SCHEMA; }
    if (std::find(ff.begin(), ff.begin() + i, ff[i]) != ff.begin() + i) { set_error("FORMAT field '%s' is selected twice", ff[i].c_str()); return BAMSCAN_ERR_SCHEMA; }
    int32_t kind;
    if (d->type == "Integer") kind = HK_ListInt32;
    else if (d->type == "Float") kind = HK_ListFloat32;
    else if (d->type == "String" || d->type == "Character") kind = HK_ListUtf8;
    else if (d->type == "Flag") { set_error("FORMAT field '%s' has Type=Flag, which a FORMAT field cannot have", d->id.c_str()); return BAMSCAN_ERR_SCHEMA; }
    else { set_error("FORMAT field '%s' has the unknown Type '%s'", d->id.c_str(), d->type.c_str()); return BAMSCAN_ERR_SCHEMA; }
    if (d->number == "0") { set_error("FORMAT field '%s' has Number=0", d->id.c_str()); return BAMSCAN_ERR_SCHEMA; }
    if (d->number != "1") {
      if (kind == HK_ListUtf8) { set_error("FORMAT field '%s': Type=%s with Number=%s is not supported by this build", d->id.c_str(), d->type.c_str(), d->number.c_str()); return BAMSCAN_ERR_UNSUPPORTED; }
      kind = kind == HK_ListInt32 ? HK_ListListInt32 : HK_ListListFloat32;
    }
    const std::string name = "format_" + d->id;
    for (const FieldDef& o : f->fields)
      if (o.name == name) { set_error("FORMAT field '%s': a column named '%s' exists already", d->id.c_str(), name.c_str()); return BAMSCAN_ERR_SCHEMA; }
    FieldDef fd{name, kind, false, {}};
    fd.metadata = {{"bio.vcf.format.number", d->number}, {"bio.vcf.format.type", d->type}, {"bio.vcf.format.description", d->description}};
    f->fields.push_back(fd);
  }
  // the sample names as a JSON array (escapes as Python's json.dumps with ensure_ascii=False)
  std::string js = "[";
  for (size_t i = 0; i < f->vcf_samples.size(); i++) {
    js += i ? ", \"" : "\"";
    for (unsigned char c : f->vcf_samples[i]) {
      if (c == '"' || c == '\\') { js += '\\'; js += (char)c; }
      else if (c == '\n') js += "\\n";
      else if (c == '\r') js += "\\r";
      else if (c == '\t') js += "\\t";
      else if (c == '\b') js += "\\b";
      else if (c == '\f') js += "\\f";
      else if (c < 0x20) { char u[8]; snprintf(u, sizeof u, "\\u%04x", c); js += u; }
      else js += (char)c;
    }
    js += '"';
  }
  js += "]";
  f->schema_metadata.push_back({"bio.vcf.samples", js});
  return BAMSCAN_OK;
}

// ---------------------------------------------------------------------------------------------
// ArrowSchema export
struct SchemaPriv {
  std::string format, name, metadata;
  std::vector<ArrowSchema> child_storage;
  std::vector<ArrowSchema*> child_ptrs;
};

static void release_schema(ArrowSchema* s) {
  if (!s || !s->release) return;
  for (int64_t i = 0; i < s->n_children; i++) if (s->children[i] && s->children[i]->release) s->children[i]->release(s->children[i]);
  delete static_cast<SchemaPriv*>(s->private_data);
  s->release = nullptr;
}

static std::string encode_metadata(const std::vector<std::pair<std::string, std::string>>& kv) {
  if (kv.empty()) return std::string();
  std::string o;
  auto put32 = [&](int32_t v) { o.append(reinterpret_cast<const char*>(&v), 4); };
  put32((int32_t)kv.size());
  for (auto& p : kv) { put32((int32_t)p.first.size()); o += p.first; put32((int32_t)p.second.size()); o += p.second; }
  return o;
}

static const char* kind_format(int32_t kind) {
  switch (kind) {
    case HK_Int32: return "i"; case HK_UInt32: return "I"; case HK_Float32: return "f"; case HK_Utf8: return "u"; case HK_Binary: return "z";
    case HK_Boolean: return "b";
    case HK_ListInt8: case HK_ListUInt8: case HK_ListInt16: case HK_ListUInt16: case HK_ListInt32: case HK_ListUInt32: case HK_ListFloat32:
    case HK_ListUtf8: case HK_ListListInt32: case HK_ListListFloat32: return "+l";
  }
  return "n";
}
static const char* list_item_format(int32_t kind) {
  switch (kind) { case HK_ListInt8: return "c"; case HK_ListUInt8: return "C"; case HK_ListInt16: return "s"; case HK_ListUInt16: return "S";
                  case HK_ListInt32: return "i"; case HK_ListUInt32: return "I"; case HK_ListFloat32: return "f"; case HK_ListUtf8: return "u";
                  case HK_ListListInt32: case HK_ListListFloat32: return "+l"; }
  return "n";
}

static void fill_schema_node(ArrowSchema* s, const char* format, const std::string& name, bool nullable,
                             const std::vector<std::pair<std::string, std::string>>& md, size_t n_children) {
  SchemaPriv* p = new SchemaPriv();
  p->format = format; p->name = name; p->metadata = encode_metadata(md);
  p->child_storage.resize(n_children); p->child_ptrs.resize(n_children);
  for (size_t i = 0; i < n_children; i++) { memset(&p->child_storage[i], 0, sizeof(ArrowSchema)); p->child_ptrs[i] = &p->child_storage[i]; }
  s->format = p->format.c_str(); s->name = p->name.c_str();
  s->metadata = p->metadata.empty() ? nullptr : p->metadata.data();
  s->flags = nullable ? ARROW_FLAG_NULLABLE : 0;
  s->n_children = (int64_t)n_children; s->children = n_children ? p->child_ptrs.data() : nullptr;
  s->dictionary = nullptr; s->release = release_schema; s->private_data = p;
}

int export_schema(const std::vector<FieldDef>& fields, const std::vector<std::pair<std::string, std::string>>& metadata, ArrowSchema* out) {
  fill_schema_node(out, "+s", "", false, metadata, fields.size());
  for (size_t i = 0; i < fields.size(); i++) {
    const FieldDef& f = fields[i];
    bool is_list = f.kind >= HK_ListInt8;
    fill_schema_node(out->children[i], kind_format(f.kind), f.name, f.nullable, f.metadata, is_list ? 1 : 0);
    const bool nested = f.kind == HK_ListListInt32 || f.kind == HK_ListListFloat32;
    if (is_list) fill_schema_node(out->children[i]->children[0], list_item_format(f.kind), "item", true, {}, nested ? 1 : 0);   // tag_registry.rs:17-19
    if (nested) fill_schema_node(out->children[i]->children[0]->children[0], f.kind == HK_ListListInt32 ? "i" : "f", "item", true, {}, 0);
  }
  return BAMSCAN_OK;
}

}  // namespace bamscan
