// writer.cu -- the device pipeline behind BamWriteExec::execute (SURVEY 8 f4) and its extern "C" entry points.
//
// == write_bam_stream (datafusion/bio-format-bam/src/write_exec.rs:278-350): header, then every batch converted to BAM
// records (batch_to_bam_records, serializer.rs:11-18) and written through the BGZF writer (writer.rs:62-113), `finish`.
// Here: Arrow buffers of a batch -> H2D -> enc_size_kernel -> scan -> enc_records_kernel into the uncompressed stream in HBM
// -> bgzf_deflate_kernel over every full 0xff00-byte member -> gather -> D2H -> write(2).  The tail that does not fill a
// member stays in HBM for the next batch; bamscan_writer_finish flushes it and appends the EOF marker.
//
// FASTQ writers (bamscan_fastq_writer_open) share everything but the encoder: no header, fq_enc_size_kernel -> scan ->
// fq_enc_records_kernel write the text into the same stream buffer, which is deflated into the same members -- or, in plain
// mode (compression 2), copied to the file as it is.
// SAM writers (bamscan_sam_writer_open) are BAM writers up to enc_size_kernel -- the same staging, row rules and reference
// lookup -- then sam_size_kernel -> scan -> sam_records_kernel write SAM lines behind the header text, and the plain path
// copies them to the file.
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "bamscan_internal.h"
#include "kernels_deflate.cuh"
#include "kernels_encode.cuh"
#include "kernels_fastq_encode.cuh"
#include "kernels_sam_encode.cuh"

namespace bamscan {

#define WCU_TRY(expr)                                                                                        \
  do {                                                                                                       \
    cudaError_t _e = (expr);                                                                                 \
    if (_e != cudaSuccess) {                                                                                 \
      set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e), __FILE__, __LINE__, #expr);           \
      return BAMSCAN_ERR_CUDA;                                                                               \
    }                                                                                                        \
  } while (0)

constexpr uint64_t SLICE_BYTES = 512ull << 20;       // uncompressed BAM bytes encoded + compressed per device pass
constexpr uint32_t SLICE_ROWS = 1u << 20;
constexpr size_t OUT_CHUNK = 16ull << 20;             // pinned D2H staging buffers (OUT_BUFS of them, drained by the file threads)
#ifndef BAMSCAN_W_FILE_THREADS
#define BAMSCAN_W_FILE_THREADS 4
#endif
#ifndef BAMSCAN_W_IN_THREADS
#define BAMSCAN_W_IN_THREADS 4
#endif
constexpr int OUT_BUFS = 12, FILE_THREADS = BAMSCAN_W_FILE_THREADS;   // 192 MB: one slice of compressed members never waits for the file threads
constexpr size_t IN_CHUNK = 8ull << 20;              // pinned H2D staging buffers (the caller's Arrow buffers are pageable)
constexpr int IN_BUFS = 2, IN_THREADS = BAMSCAN_W_IN_THREADS;

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
static const bool g_wtrace = getenv("BAMSCAN_WRITER_TRACE") != nullptr;
#define WTRACE(...) do { if (g_wtrace) fprintf(stderr, __VA_ARGS__); } while (0)

struct DevBuf {
  void* p = nullptr; size_t cap = 0;
  int reserve(size_t n) {
    if (n <= cap) return BAMSCAN_OK;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    const size_t want = n + n / 4 + 4096;
    if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); set_error("cudaMalloc(%zu) failed in the BAM writer", want); return BAMSCAN_ERR_CUDA; }
    cap = want;
    return BAMSCAN_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct WTag { int col; int32_t kind; uint8_t tag[2], sam_type, subtype; };

// Device buffers, pinned staging, stream and events of a writer.  One set per device is kept between writers (cudaMalloc /
// cudaHostAlloc / cudaFree of a few GB cost more than writing a few million records).
struct WriterRes {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[4] = {}, ev2[2] = {}, in_free[IN_BUFS] = {};
  DevBuf ref_blob, ref_off, ref_ids, in, stream_buf, rec_len, ref_pairs, cig_bin, cig_tmp, rec_off, tile_sums, slots, sizes, offsets, packed, tok, small;
  uint8_t* h_out[OUT_BUFS] = {};         // pinned; filled by D2H, written to the file by the file threads
  uint8_t* h_in[IN_BUFS] = {};           // pinned; the caller's buffers are copied here by IN_THREADS host threads, then H2D
  uint64_t* h_small = nullptr;           // pinned: tile sums, totals, error words
  bool ready = false;
  void destroy() {
    for (DevBuf* b : {&ref_blob, &ref_off, &ref_ids, &in, &stream_buf, &rec_len, &ref_pairs, &cig_bin, &cig_tmp, &rec_off, &tile_sums, &slots, &sizes, &offsets, &packed, &tok, &small}) b->release();
    for (auto& b : h_out) { if (b) cudaFreeHost(b); b = nullptr; }
    for (auto& b : h_in) { if (b) cudaFreeHost(b); b = nullptr; }
    if (h_small) { cudaFreeHost(h_small); h_small = nullptr; }
    for (auto& e : ev) { if (e) cudaEventDestroy(e); e = nullptr; }
    for (auto& e : ev2) { if (e) cudaEventDestroy(e); e = nullptr; }
    for (auto& e : in_free) { if (e) cudaEventDestroy(e); e = nullptr; }
    if (stream) { cudaStreamDestroy(stream); stream = nullptr; }
    ready = false;
  }
};
static std::mutex g_res_mu;
static WriterRes g_res_pool[64];

}  // namespace bamscan

using namespace bamscan;

struct BamWriter : bamscan::WriterRes {
  int fd = -1;
  std::string path;
  int device = 0;
  bool zero_based = true, cigar_binary = false, finished = false;
  int compression = 0;
  ScanFormat format = FMT_BAM;
  bool plain = false;                    // FASTQ compression 2, SAM: the text goes to the file as it is (no BGZF, no EOF marker)
  int col[11] = {};                      // BAM, SAM: name chrom start flags cigar mapq mate_chrom mate_start seq qual tlen;
                                         // FASTQ: name description (-1: absent) sequence quality_scores
  std::vector<WTag> tags;
  int n_cols = 0;
  int n_ref = 0;
  uint32_t slice_rows = SLICE_ROWS;      // rows per device pass (shrinks for long reads)
  bool src_on_device = false;            // bamscan_writer_write_device: the batch's buffers are device pointers
  uint64_t pending = 0;                  // bytes of the uncompressed stream waiting at the front of stream_buf (header, tails)
  uint64_t in_seq = 0;
  // file threads: pwrite(2) of the pieces of a staging buffer runs beside the GPU work of the next slice
  struct FileJob { int slot; size_t at, bytes; uint64_t file_off; };
  std::thread file_thread[FILE_THREADS];
  std::mutex mu;
  std::condition_variable cv;
  std::deque<FileJob> file_q;
  int out_busy[OUT_BUFS] = {};           // outstanding pieces per buffer
  uint64_t file_off = 0;
  bool file_stop = false, file_failed = false;
  int n_sms = 148;
  BamWriteStats st = {};
};

namespace bamscan {

static const char* enc_err_text(uint32_t code) {
  switch (code) {
    case enc::ENC_ERR_FLAGS: return "Flag value does not fit into 16-bit SAM flags";
    case enc::ENC_ERR_CIGAR: return "Failed to parse CIGAR";
    case enc::ENC_ERR_CIGAR_LEN: return "CIGAR op length does not fit 28 bits";
    case enc::ENC_ERR_CIGAR_OPS: return "more than 65535 CIGAR ops (CG-tag overflow) is not supported by this build";
    case enc::ENC_ERR_QUAL_LEN: return "sequence-quality scores length mismatch";
    case enc::ENC_ERR_NAME_LEN: return "read name longer than 254 bytes";
    case enc::ENC_ERR_TAG_RANGE: return "tag value does not fit its SAM type";
    case enc::ENC_ERR_TAG_HEX: return "Invalid SAM hex tag value";
    case enc::ENC_ERR_TAG_CHAR: return "Character tags must be a single ASCII byte";
    case enc::ENC_ERR_CIGAR_BIN: return "Failed to decode binary CIGAR";
    case enc::ENC_ERR_REC_LEN: return "record larger than 2 GiB";
    case enc::ENC_ERR_POS: return "position does not fit the 32-bit BAM field";
    case samenc::SAM_ERR_QNAME: return "invalid QNAME (SAM allows 1 to 254 characters of [!-?A-~])";
    case samenc::SAM_ERR_SEQ: return "invalid SEQ (SAM allows [A-Za-z=.])";
    case samenc::SAM_ERR_QUAL: return "invalid QUAL (a quality character above '~')";
    case samenc::SAM_ERR_TAG_Z: return "invalid Z tag value (SAM allows [ !-~])";
    case samenc::SAM_ERR_TAG_A: return "invalid A tag value (SAM allows one character of [!-~])";
    case samenc::SAM_ERR_LINE_LEN: return "SAM line larger than 2 GiB";
    case samenc::SAM_ERR_INTERNAL: return "internal error: a SAM line does not have its sized length";
    default: return "encode error";
  }
}

// error class of an encoder code: tag value checks are schema errors, CG-tag overflow is unsupported, the rest format errors
static int enc_err_class(uint32_t code) {
  return (code == enc::ENC_ERR_TAG_RANGE || code == enc::ENC_ERR_TAG_HEX || code == enc::ENC_ERR_TAG_CHAR) ? BAMSCAN_ERR_SCHEMA
         : code == enc::ENC_ERR_CIGAR_OPS ? BAMSCAN_ERR_UNSUPPORTED : BAMSCAN_ERR_FORMAT;
}

static std::map<std::string, std::string> parse_metadata(const char* md) {
  std::map<std::string, std::string> out;
  if (!md) return out;
  int32_t n; memcpy(&n, md, 4); md += 4;
  for (int32_t i = 0; i < n; i++) {
    int32_t kl; memcpy(&kl, md, 4); md += 4;
    std::string k(md, (size_t)kl); md += kl;
    int32_t vl; memcpy(&vl, md, 4); md += 4;
    std::string v(md, (size_t)vl); md += vl;
    out[k] = v;
  }
  return out;
}

static int32_t kind_of_format(const ArrowSchema* c) {
  const std::string f = c->format ? c->format : "";
  if (f == "i") return HK_Int32;
  if (f == "I") return HK_UInt32;
  if (f == "f") return HK_Float32;
  if (f == "u") return HK_Utf8;
  if (f == "z") return HK_Binary;
  if (f == "c") return enc::WK_Int8;          // scalar tag columns only (the scan itself never produces these)
  if (f == "C") return enc::WK_UInt8;
  if (f == "s") return enc::WK_Int16;
  if (f == "S") return enc::WK_UInt16;
  if (f == "l") return enc::WK_Int64;
  if (f == "L") return enc::WK_UInt64;
  if (f == "g") return enc::WK_Float64;
  if (f == "+l" && c->n_children == 1 && c->children[0]->format) {
    const std::string e = c->children[0]->format;
    if (e == "c") return HK_ListInt8;
    if (e == "C") return HK_ListUInt8;
    if (e == "s") return HK_ListInt16;
    if (e == "S") return HK_ListUInt16;
    if (e == "i") return HK_ListInt32;
    if (e == "I") return HK_ListUInt32;
    if (e == "f") return HK_ListFloat32;
  }
  return 0;
}

static int writer_flush_members(BamWriter* w, uint64_t total, bool final_flush);
static int writer_open_device(BamWriter* w, int device_id);
static int writer_open_file(BamWriter* w, const char* output_path);

static int writer_open_impl(const char* output_path, const char* sam_header_text, int32_t n_ref, const char* const* ref_names,
                            const int32_t* ref_lengths, const ArrowSchema* schema, const BamWriteOptions* options, BamWriter** out,
                            ScanFormat format = FMT_BAM) {
  if (!output_path || !schema || !out || (n_ref > 0 && (!ref_names || !ref_lengths))) { set_error("bamscan_writer_open: null argument"); return BAMSCAN_ERR_INVALID; }
  BamWriteOptions opt;
  memset(&opt, 0, sizeof opt);
  opt.coordinate_system_zero_based = 1;
  if (options) memcpy(&opt, options, std::min<size_t>(sizeof opt, options->struct_size ? options->struct_size : sizeof opt));
  if (!schema->format || strcmp(schema->format, "+s") != 0) { set_error("bamscan_writer_open: input_schema must be a struct"); return BAMSCAN_ERR_INVALID; }
  std::unique_ptr<BamWriter, void (*)(BamWriter*)> w(new BamWriter(), [](BamWriter* p) { bamscan_writer_free(p); });   // (error paths give the pooled resources back)
  w->path = output_path; w->device = opt.device_id; w->zero_based = opt.coordinate_system_zero_based != 0; w->compression = opt.compression;
  w->format = format; w->plain = format == FMT_SAM;        // (SAM: plain text, `compression` is not read)
  w->n_cols = (int)schema->n_children;
  // columns by name (sam_record_serializer.rs:27-37: every core column is required; `end` is not read)
  static const char* const names[11] = {"name", "chrom", "start", "flags", "cigar", "mapping_quality", "mate_chrom", "mate_start", "sequence", "quality_scores", "template_length"};
  static const int32_t want[11] = {HK_Utf8, HK_Utf8, HK_UInt32, HK_UInt32, HK_Utf8, HK_UInt32, HK_Utf8, HK_UInt32, HK_Utf8, HK_Utf8, HK_Int32};
  for (int k = 0; k < 11; k++) {
    int idx = -1;
    for (int64_t c = 0; c < schema->n_children; c++) if (schema->children[c]->name && strcmp(schema->children[c]->name, names[k]) == 0) { idx = (int)c; break; }
    if (idx < 0) { set_error("Required column '%s' not found in batch", names[k]); return BAMSCAN_ERR_SCHEMA; }
    const int32_t kind = kind_of_format(schema->children[idx]);
    if (k == 4 && kind == HK_Binary) w->cigar_binary = true;
    else if (kind != want[k]) { set_error("Column '%s' must be %s type", names[k], want[k] == HK_Utf8 ? "String" : want[k] == HK_UInt32 ? "UInt32" : "Int32"); return BAMSCAN_ERR_SCHEMA; }
    w->col[k] = idx;
  }
  // tag columns (build_tag_column_map, sam_record_serializer.rs:281-298; type letters: sam_tag_io.rs:127-141, 206-235)
  for (int t = 0; t < opt.n_tag_fields && opt.tag_fields; t++) {
    const char* tn = opt.tag_fields[t];
    int idx = -1;
    for (int64_t c = 0; c < schema->n_children; c++) if (schema->children[c]->name && strcmp(schema->children[c]->name, tn) == 0) { idx = (int)c; break; }
    if (idx < 0) continue;
    const auto md = parse_metadata(schema->children[idx]->metadata);
    if (!md.count("bio.bam.tag.tag") || strlen(tn) != 2) continue;
    auto alpha = [](char c) { return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z'); };
    if (format == FMT_SAM && !(alpha(tn[0]) && (alpha(tn[1]) || (tn[1] >= '0' && tn[1] <= '9')))) {   // the SAM reader refuses other names
      set_error("tag column '%s': a SAM tag name must match [A-Za-z][A-Za-z0-9]", tn); return BAMSCAN_ERR_SCHEMA;
    }
    std::string spec = md.count("bio.bam.tag.type") ? md.at("bio.bam.tag.type") : "Z";
    WTag g; g.col = idx; g.kind = kind_of_format(schema->children[idx]); g.tag[0] = (uint8_t)tn[0]; g.tag[1] = (uint8_t)tn[1]; g.subtype = 0;
    if (spec.size() == 1) g.sam_type = (uint8_t)spec[0];
    else if (spec.size() == 3 && spec[0] == 'B' && spec[1] == ':' && strchr("cCsSiIf", spec[2])) { g.sam_type = 'B'; g.subtype = (uint8_t)spec[2]; }
    else { set_error("Invalid SAM tag type metadata: '%s'", spec.c_str()); return BAMSCAN_ERR_SCHEMA; }
    if (!g.kind) { set_error("tag column '%s': Arrow type '%s' is not supported by this build (integers of 8 to 64 bits, Float32 / Float64, Utf8, List of 8/16/32-bit integers or Float32)", tn, schema->children[idx]->format); return BAMSCAN_ERR_UNSUPPORTED; }
    const bool is_int = g.kind == HK_Int32 || g.kind == HK_UInt32 || (g.kind >= enc::WK_Int8 && g.kind <= enc::WK_UInt64);
    const bool is_list = g.kind >= HK_ListInt8 && g.kind <= HK_ListFloat32;
    const char st = (char)g.sam_type;
    bool ok;
    if (strchr("cCsSiI", st)) ok = is_int;
    else if (st == 'f') ok = g.kind == HK_Float32 || g.kind == enc::WK_Float64;
    else if (st == 'Z' || st == 'H') ok = g.kind == HK_Utf8;
    else if (st == 'A') ok = g.kind == HK_Utf8 || is_int;
    else if (st == 'B') {
      ok = is_list;
      if (ok && !g.subtype) g.subtype = (uint8_t)"cCsSiIf"[g.kind - HK_ListInt8];
      if (ok && g.subtype == 'f' && g.kind != HK_ListFloat32) ok = false;
      if (ok && g.subtype != 'f' && g.kind == HK_ListFloat32) ok = false;
    } else {                                  // unknown letter: strings pass as Z, every other column is dropped (sam_tag_io.rs:227-233)
      if (g.kind != HK_Utf8) continue;
      g.sam_type = 'Z'; ok = true;
    }
    if (!ok) { set_error("Tag value type mismatch: column '%s' (Arrow format '%s') cannot be written as SAM type '%s'", tn, schema->children[idx]->format, spec.c_str()); return BAMSCAN_ERR_SCHEMA; }
    if ((int)w->tags.size() >= enc::MAX_WTAGS) { set_error("more than %d tag columns are not supported by the writer", enc::MAX_WTAGS); return BAMSCAN_ERR_UNSUPPORTED; }
    w->tags.push_back(g);
  }
  int rc;
  if ((rc = writer_open_device(w.get(), opt.device_id))) return rc;
  // reference dictionary, sorted bytewise; a later duplicate wins like the reference's HashMap collect
  {
    std::map<std::string, int32_t> m;
    for (int32_t i = 0; i < n_ref; i++) m[ref_names[i]] = i;
    std::string blob; std::vector<int32_t> off{0}, ids;
    for (auto& kv : m) { blob += kv.first; off.push_back((int32_t)blob.size()); ids.push_back(kv.second); }
    w->n_ref = (int)ids.size();
    if ((rc = w->ref_blob.reserve(blob.size() + 16)) || (rc = w->ref_off.reserve(off.size() * 4)) || (rc = w->ref_ids.reserve(ids.size() * 4 + 4))) return rc;
    if (!blob.empty()) WCU_TRY(cudaMemcpy(w->ref_blob.p, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    WCU_TRY(cudaMemcpy(w->ref_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice));
    if (!ids.empty()) WCU_TRY(cudaMemcpy(w->ref_ids.p, ids.data(), ids.size() * 4, cudaMemcpyHostToDevice));
  }
  // BAM header bytes open the uncompressed stream (bam::io::Writer::write_header); a SAM file starts with the header text as given
  std::string hdr("BAM\1", 4);
  if (format == FMT_SAM) { hdr = sam_header_text ? sam_header_text : ""; w->st.bam_bytes = hdr.size(); }
  else {
    const std::string text = sam_header_text ? sam_header_text : "";
    auto put32 = [&](int32_t v) { hdr.append(reinterpret_cast<const char*>(&v), 4); };
    put32((int32_t)text.size()); hdr += text; put32(n_ref);
    for (int32_t i = 0; i < n_ref; i++) { const std::string n = ref_names[i]; put32((int32_t)n.size() + 1); hdr += n; hdr.push_back('\0'); put32(ref_lengths[i]); }
  }
  if ((rc = w->stream_buf.reserve(hdr.size() + SLICE_BYTES + 65536))) return rc;
  if (!hdr.empty()) WCU_TRY(cudaMemcpy(w->stream_buf.p, hdr.data(), hdr.size(), cudaMemcpyHostToDevice));
  w->pending = hdr.size();
  if ((rc = writer_open_file(w.get(), output_path))) return rc;
  *out = w.release();
  return BAMSCAN_OK;
}

// Device, pooled resources and the CRC table of the deflate kernel: the part of opening a writer that needs the GPU.
static int writer_open_device(BamWriter* w, int device_id) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); set_error("bamscan_writer_open: no CUDA device (this library has no CPU path)"); return BAMSCAN_ERR_CUDA; }
  if (device_id < 0 || device_id >= ndev) { set_error("device_id %d out of range (%d devices)", device_id, ndev); return BAMSCAN_ERR_INVALID; }
  WCU_TRY(cudaSetDevice(device_id));
  cudaDeviceProp prop;
  WCU_TRY(cudaGetDeviceProperties(&prop, device_id));
  w->n_sms = prop.multiProcessorCount;
  {
    std::lock_guard<std::mutex> lk(g_res_mu);
    WriterRes& pooled = g_res_pool[device_id & 63];
    if (pooled.ready) { static_cast<WriterRes&>(*w) = pooled; pooled = WriterRes(); }
  }
  if (!w->ready) {
    WCU_TRY(cudaStreamCreateWithFlags(&w->stream, cudaStreamNonBlocking));
    for (auto& e : w->ev) WCU_TRY(cudaEventCreate(&e));
    for (auto& e : w->ev2) WCU_TRY(cudaEventCreate(&e));
    for (auto& b : w->h_out) WCU_TRY(cudaHostAlloc((void**)&b, OUT_CHUNK, cudaHostAllocDefault));
    for (auto& b : w->h_in) WCU_TRY(cudaHostAlloc((void**)&b, IN_CHUNK, cudaHostAllocDefault));
    for (auto& e : w->in_free) WCU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    WCU_TRY(cudaHostAlloc((void**)&w->h_small, 1 << 16, cudaHostAllocDefault));
    w->ready = true;
  }
  {
    auto mulmod = [](uint32_t a, uint32_t b) { uint32_t p = 0; for (int i = 0; i < 32; i++) { if (b & 0x80000000u) p ^= a; a = (a >> 1) ^ ((a & 1u) ? 0xEDB88320u : 0u); b <<= 1; } return p; };
    uint32_t tab[18];
    tab[0] = 0x00800000u;
    for (int j = 1; j < 18; j++) tab[j] = mulmod(tab[j - 1], tab[j - 1]);
    WCU_TRY(cudaMemcpyToSymbol(dfl::c_xpow8, tab, sizeof tab));
    WCU_TRY(cudaFuncSetAttribute(dfl::bgzf_deflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(dfl::Smem)));
  }
  return BAMSCAN_OK;
}

// Creates the output file and starts the file threads.
static int writer_open_file(BamWriter* w, const char* output_path) {
  w->fd = ::open(output_path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
  if (w->fd < 0) { set_error("Failed to create output file: %s", output_path); return BAMSCAN_ERR_IO; }
  {
    BamWriter* wp = w;
    for (auto& th : wp->file_thread) th = std::thread([wp] {
      for (;;) {
        BamWriter::FileJob job;
        {
          std::unique_lock<std::mutex> lk(wp->mu);
          wp->cv.wait(lk, [wp] { return wp->file_stop || !wp->file_q.empty(); });
          if (wp->file_q.empty()) return;
          job = wp->file_q.front(); wp->file_q.pop_front();
        }
        size_t done = 0;
        while (done < job.bytes && !wp->file_failed) {
          const ssize_t k = ::pwrite(wp->fd, wp->h_out[job.slot] + job.at + done, job.bytes - done, (off_t)(job.file_off + done));
          if (k <= 0) { wp->file_failed = true; break; }
          done += (size_t)k;
        }
        { std::lock_guard<std::mutex> lk(wp->mu); wp->out_busy[job.slot]--; }
        wp->cv.notify_all();
      }
    });
  }
  return BAMSCAN_OK;
}

// FASTQ writer: columns by name (name, sequence, quality_scores required, description optional, all Utf8; any other column is
// ignored), no header bytes, compression 0 / 1 (BGZF) or 2 (plain text).
static int fastq_writer_open_impl(const char* output_path, const ArrowSchema* schema, const BamWriteOptions* options, BamWriter** out) {
  if (!output_path || !schema || !out) { set_error("bamscan_fastq_writer_open: null argument"); return BAMSCAN_ERR_INVALID; }
  BamWriteOptions opt;
  memset(&opt, 0, sizeof opt);
  if (options) memcpy(&opt, options, std::min<size_t>(sizeof opt, options->struct_size ? options->struct_size : sizeof opt));
  if (!schema->format || strcmp(schema->format, "+s") != 0) { set_error("bamscan_fastq_writer_open: input_schema must be a struct"); return BAMSCAN_ERR_INVALID; }
  if (opt.compression < 0 || opt.compression > 2) { set_error("bamscan_fastq_writer_open: compression %d (0: BGZF, 1: BGZF stored blocks, 2: plain text)", opt.compression); return BAMSCAN_ERR_INVALID; }
  std::unique_ptr<BamWriter, void (*)(BamWriter*)> w(new BamWriter(), [](BamWriter* p) { bamscan_writer_free(p); });
  w->path = output_path; w->device = opt.device_id; w->compression = opt.compression;
  w->format = FMT_FASTQ; w->plain = opt.compression == 2;
  w->n_cols = (int)schema->n_children;
  static const char* const names[4] = {"name", "description", "sequence", "quality_scores"};
  for (int k = 0; k < 4; k++) {
    int idx = -1;
    for (int64_t c = 0; c < schema->n_children; c++) if (schema->children[c]->name && strcmp(schema->children[c]->name, names[k]) == 0) { idx = (int)c; break; }
    if (idx < 0 && k == 1) { w->col[k] = -1; continue; }
    if (idx < 0) { set_error("Required column '%s' not found in batch", names[k]); return BAMSCAN_ERR_SCHEMA; }
    if (kind_of_format(schema->children[idx]) != HK_Utf8) { set_error("Column '%s' must be Utf8", names[k]); return BAMSCAN_ERR_SCHEMA; }
    w->col[k] = idx;
  }
  int rc;
  if ((rc = writer_open_device(w.get(), opt.device_id))) return rc;
  if ((rc = w->stream_buf.reserve(SLICE_BYTES + 65536))) return rc;
  w->pending = 0;
  if ((rc = writer_open_file(w.get(), output_path))) return rc;
  *out = w.release();
  return BAMSCAN_OK;
}

// H2D of one buffer slice; returns the device address of its first byte.  Large slices go through the pinned ring: IN_THREADS
// host threads copy a chunk into a pinned buffer, one cudaMemcpyAsync sends it on (pageable H2D would be staged by the
// driver on one thread at a fraction of the link rate).
static int stage(BamWriter* w, size_t* cursor, const void* src, size_t bytes, uint8_t** dev) {
  if (w->src_on_device) { *dev = const_cast<uint8_t*>(static_cast<const uint8_t*>(src)); return BAMSCAN_OK; }   // the batch already lives in HBM
  const size_t at = (*cursor + 15) & ~size_t(15);
  *dev = static_cast<uint8_t*>(w->in.p) + at;
  *cursor = at + bytes;
  w->st.arrow_bytes += bytes;
  const uint8_t* s = static_cast<const uint8_t*>(src);
  if (bytes >= (1u << 20)) {
    // a source that is already page-locked (e.g. the arenas the scan hands its batches out in) goes by DMA as it stands; the
    // stream is synchronised before bamscan_writer_write returns, so the caller's buffer outlives the copy
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, src) == cudaSuccess && at.type == cudaMemoryTypeHost) {
      WCU_TRY(cudaMemcpyAsync(*dev, s, bytes, cudaMemcpyHostToDevice, w->stream));
      return BAMSCAN_OK;
    }
    cudaGetLastError();
  }
  for (size_t done = 0; done < bytes;) {
    const size_t nb = std::min(IN_CHUNK, bytes - done);
    const int slot = (int)(w->in_seq % IN_BUFS);
    if (w->in_seq >= (uint64_t)IN_BUFS) WCU_TRY(cudaEventSynchronize(w->in_free[slot]));
    uint8_t* h = w->h_in[slot];
    if (nb >= (4u << 20)) {
      std::thread th[IN_THREADS];
      const size_t per = (nb + IN_THREADS - 1) / IN_THREADS;
      for (int t = 0; t < IN_THREADS; t++) {
        const size_t b = std::min(nb, per * t), e = std::min(nb, b + per);
        th[t] = std::thread([=] { if (e > b) memcpy(h + b, s + done + b, e - b); });
      }
      for (auto& t : th) t.join();
    } else memcpy(h, s + done, nb);
    WCU_TRY(cudaMemcpyAsync(*dev + done, h, nb, cudaMemcpyHostToDevice, w->stream));
    WCU_TRY(cudaEventRecord(w->in_free[slot], w->stream));
    w->in_seq++;
    done += nb;
  }
  return BAMSCAN_OK;
}

struct HostCol { const ArrowArray* a; int64_t off; };     // off = struct offset + child offset

// first and last entry of an offsets buffer (a device batch: two 4-byte reads from HBM)
static bool off_ends(const BamWriter* w, const void* offsets, int64_t i0, int64_t i1, int32_t* first, int32_t* last) {
  const int32_t* o = static_cast<const int32_t*>(offsets);
  if (!w->src_on_device) { *first = o[i0]; *last = o[i1]; return true; }
  return cudaMemcpy(first, o + i0, 4, cudaMemcpyDeviceToHost) == cudaSuccess && cudaMemcpy(last, o + i1, 4, cudaMemcpyDeviceToHost) == cudaSuccess;
}
static size_t utf8_bytes(const BamWriter* w, const HostCol& c, int64_t n) {
  int32_t a = 0, b = 0;
  off_ends(w, c.a->buffers[1], c.off, c.off + n, &a, &b);
  return (size_t)(b - a) + (size_t)(n + 1) * 4 + (size_t)(n / 8 + 2) + 64;
}

static int stage_validity(BamWriter* w, size_t* cur, const HostCol& c, int64_t n, const uint8_t** out) {
  *out = nullptr;
  const uint8_t* v = static_cast<const uint8_t*>(c.a->buffers[0]);
  if (!v || c.a->null_count == 0) return BAMSCAN_OK;
  if (w->src_on_device) { *out = v; return BAMSCAN_OK; }
  const int64_t b0 = c.off >> 3, b1 = (c.off + n + 7) >> 3;
  uint8_t* d; int rc = stage(w, cur, v + b0, (size_t)(b1 - b0), &d);
  if (rc) return rc;
  *out = d - b0;                                          // indexable by (array offset + row)
  return BAMSCAN_OK;
}
static int stage_utf8(BamWriter* w, size_t* cur, const HostCol& c, int64_t n, enc::Utf8Col* out) {
  const int32_t* o = static_cast<const int32_t*>(c.a->buffers[1]);
  const uint8_t* data = static_cast<const uint8_t*>(c.a->buffers[2]);
  uint8_t* d; int rc;
  if ((rc = stage(w, cur, o + c.off, (size_t)(n + 1) * 4, &d))) return rc;
  out->off = reinterpret_cast<const int32_t*>(d) - c.off;
  int32_t first = 0, last = 0;
  if (!off_ends(w, o, c.off, c.off + n, &first, &last)) { set_error("bamscan_writer_write_device: cannot read the offsets of a device batch"); return BAMSCAN_ERR_CUDA; }
  if ((rc = stage(w, cur, data ? data + first : nullptr, data ? (size_t)(last - first) : 0, &d))) return rc;
  out->data = d - first;
  out->base = c.off;
  return stage_validity(w, cur, c, n, &out->valid);
}
static int stage_prim(BamWriter* w, size_t* cur, const HostCol& c, int64_t n, enc::PrimCol* out, size_t es = 4) {
  const uint8_t* v = static_cast<const uint8_t*>(c.a->buffers[1]);
  uint8_t* d; int rc;
  if ((rc = stage(w, cur, v + (size_t)c.off * es, (size_t)n * es, &d))) return rc;
  out->values = reinterpret_cast<const uint32_t*>(d - (size_t)c.off * es);
  out->base = c.off;
  return stage_validity(w, cur, c, n, &out->valid);
}

// Byte count of a slice from the record lengths in rec_len: tile sums on the device, exclusive tile offsets into h_small[0 ..
// n_tiles) on the host.  The slice's error words come back beside them (h_small + 4096), read by the caller.
static int sum_lengths(BamWriter* w, uint32_t rows, const uint32_t* d_err, uint64_t* total) {
  const uint32_t n_tiles = (rows + 4095) / 4096;
  unsigned long long* d_tiles = static_cast<unsigned long long*>(w->tile_sums.p);
  dfl::len_tile_sums_kernel<<<n_tiles, 256, 0, w->stream>>>(static_cast<uint32_t*>(w->rec_len.p), rows, d_tiles);
  w->st.kernel_launches += 1;
  WCU_TRY(cudaMemcpyAsync(w->h_small, d_tiles, (size_t)n_tiles * 8, cudaMemcpyDeviceToHost, w->stream));
  WCU_TRY(cudaMemcpyAsync(w->h_small + 4096, d_err, 16, cudaMemcpyDeviceToHost, w->stream));
  WCU_TRY(cudaStreamSynchronize(w->stream));
  uint64_t t = 0;
  for (uint32_t k = 0; k < n_tiles; k++) { const uint64_t s = w->h_small[k]; w->h_small[k] = t; t += s; }
  *total = t;
  return BAMSCAN_OK;
}

// 64-bit record offsets rec_off[0 .. rows] in the stream buffer, behind its pending bytes (grown when one slice does not fit).
static int place_records(BamWriter* w, uint32_t rows, uint64_t total) {
  const uint32_t n_tiles = (rows + 4095) / 4096;
  unsigned long long* d_tiles = static_cast<unsigned long long*>(w->tile_sums.p);
  if (w->pending + total + 65536 > w->stream_buf.cap) {    // one record larger than a slice: grow, keeping the pending bytes
    DevBuf bigger;
    int rc;
    if ((rc = bigger.reserve(w->pending + total + 65536))) return rc;
    WCU_TRY(cudaMemcpyAsync(bigger.p, w->stream_buf.p, w->pending, cudaMemcpyDeviceToDevice, w->stream));
    WCU_TRY(cudaStreamSynchronize(w->stream));
    w->stream_buf.release(); w->stream_buf = bigger;
  }
  WCU_TRY(cudaMemcpyAsync(d_tiles + n_tiles + 1, w->h_small, (size_t)n_tiles * 8, cudaMemcpyHostToDevice, w->stream));
  dfl::len_offsets_kernel<<<n_tiles, 256, 0, w->stream>>>(static_cast<uint32_t*>(w->rec_len.p), rows, d_tiles + n_tiles + 1, w->pending,
                                                         static_cast<unsigned long long*>(w->rec_off.p));
  w->st.kernel_launches += 1;
  w->h_small[6000] = w->pending + total;                    // (rows % 4096 == 0: no tile of the kernel above owns element `rows`)
  WCU_TRY(cudaMemcpyAsync(static_cast<unsigned long long*>(w->rec_off.p) + rows, w->h_small + 6000, 8, cudaMemcpyHostToDevice, w->stream));
  return BAMSCAN_OK;
}

static const char* fq_err_text(uint32_t code) {
  switch (code) {
    case fqenc::FQ_ERR_NULL_NAME: return "name is NULL";
    case fqenc::FQ_ERR_NULL_SEQ: return "sequence is NULL";
    case fqenc::FQ_ERR_NULL_QUAL: return "quality_scores is NULL";
    case fqenc::FQ_ERR_EOL_NAME: return "line break in name";
    case fqenc::FQ_ERR_WS_NAME: return "space or tab in name";
    case fqenc::FQ_ERR_EOL_DESC: return "line break in description";
    case fqenc::FQ_ERR_EOL_SEQ: return "line break in sequence";
    case fqenc::FQ_ERR_EOL_QUAL: return "line break in quality_scores";
    case fqenc::FQ_ERR_REC_LEN: return "record larger than 2 GiB";
    default: return "encode error";
  }
}

// The FASTQ branch of bamscan_writer_write(_device): stage the four Utf8 columns, then per slice of rows sizes -> offsets ->
// text -> members (or, plain, the file).
static int fastq_write_impl(BamWriter* w, const ArrowArray* batch, int64_t n) {
  auto hc = [&](int idx) { return HostCol{batch->children[idx], batch->offset + batch->children[idx]->offset}; };
  for (int k = 0; k < 4; k++) {
    if (w->col[k] < 0) continue;
    const ArrowArray* a = batch->children[w->col[k]];
    if (!a || !a->buffers || a->n_buffers < 3 || !a->buffers[1] || a->length + a->offset < n + batch->offset) {
      set_error("bamscan_writer_write: column %d of the batch does not have the layout of the writer's input schema", w->col[k]);
      return BAMSCAN_ERR_INVALID;
    }
  }
  size_t need = 4096;
  if (!w->src_on_device) for (int k = 0; k < 4; k++) if (w->col[k] >= 0) need += utf8_bytes(w, hc(w->col[k]), n);
  int rc;
  const double t_w0 = now_ms();
  if ((rc = w->in.reserve(need))) return rc;
  fqenc::FqArgs A;
  memset(&A, 0, sizeof A);
  size_t cur = 0;
  A.has_desc = w->col[1] >= 0;
  if ((rc = stage_utf8(w, &cur, hc(w->col[0]), n, &A.name)) || (A.has_desc && (rc = stage_utf8(w, &cur, hc(w->col[1]), n, &A.desc))) ||
      (rc = stage_utf8(w, &cur, hc(w->col[2]), n, &A.seq)) || (rc = stage_utf8(w, &cur, hc(w->col[3]), n, &A.qual)))
    return rc;
  WTRACE("[writer] FASTQ batch of %lld rows: staged %.1f MB in %.1f ms\n", (long long)n, cur / 1e6, now_ms() - t_w0);
  if ((rc = w->small.reserve(4096))) return rc;
  uint32_t* d_err = static_cast<uint32_t*>(w->small.p);
  const uint32_t* h_err = reinterpret_cast<const uint32_t*>(w->h_small + 4096);
  int64_t r0 = 0;
  uint32_t want_rows = w->slice_rows;
  while (r0 < n) {
    const uint32_t rows = (uint32_t)std::min<int64_t>(want_rows, n - r0);
    if ((rc = w->rec_len.reserve((size_t)rows * 4)) || (rc = w->rec_off.reserve(((size_t)rows + 1) * 8)) || (rc = w->tile_sums.reserve(((size_t)rows / 4096 + 2) * 16)))
      return rc;
    A.row0 = (uint32_t)r0; A.n_rows = rows;
    WCU_TRY(cudaEventRecord(w->ev[0], w->stream));
    WCU_TRY(cudaMemsetAsync(d_err, 0, 16, w->stream));
    fqenc::fq_enc_size_kernel<<<(rows + 255) / 256, 256, 0, w->stream>>>(A, static_cast<uint32_t*>(w->rec_len.p), d_err);
    w->st.kernel_launches += 1;
    uint64_t total = 0;
    if ((rc = sum_lengths(w, rows, d_err, &total))) return rc;
    if (h_err[0]) { set_error("FASTQ write error: row %u: %s", h_err[1], fq_err_text(h_err[0])); return BAMSCAN_ERR_FORMAT; }
    if (total > SLICE_BYTES && rows > 1) {                   // long reads: fewer rows per pass
      want_rows = std::max<uint32_t>(1, (uint32_t)((double)rows * (double)SLICE_BYTES / (double)total * 0.9));
      w->slice_rows = want_rows;
      continue;
    }
    if ((rc = place_records(w, rows, total))) return rc;
    const unsigned long long* d_off = static_cast<const unsigned long long*>(w->rec_off.p);
    uint8_t* d_out = static_cast<uint8_t*>(w->stream_buf.p);
    if (total / rows > 2048) fqenc::fq_enc_records_kernel<32><<<(rows * 32 + 255) / 256, 256, 0, w->stream>>>(A, d_off, d_out, d_err);   // long reads: a warp per row
    else fqenc::fq_enc_records_kernel<8><<<(((rows + 3) / 4) * 32 + 255) / 256, 256, 0, w->stream>>>(A, d_off, d_out, d_err);
    w->st.kernel_launches += 1;
    WCU_TRY(cudaEventRecord(w->ev[1], w->stream));
    WCU_TRY(cudaMemcpyAsync(w->h_small + 4096, d_err, 16, cudaMemcpyDeviceToHost, w->stream));
    WCU_TRY(cudaStreamSynchronize(w->stream));
    if (h_err[0]) { set_error("FASTQ write error: row %u: %s", h_err[1], fq_err_text(h_err[0])); return BAMSCAN_ERR_FORMAT; }
    { float ms = 0; cudaEventElapsedTime(&ms, w->ev[0], w->ev[1]); w->st.ms_encode += ms; w->st.ms_total += ms; }
    w->st.rows += rows; w->st.bam_bytes += total;
    const double t_f0 = now_ms();
    if ((rc = writer_flush_members(w, w->pending + total, false))) return rc;
    WTRACE("[writer] FASTQ slice of %u rows: encode done at +%.1f ms, flushed in %.1f ms\n", rows, t_f0 - t_w0, now_ms() - t_f0);
    r0 += rows;
  }
  return BAMSCAN_OK;
}

static int writer_write_impl(BamWriter* w, const ArrowArray* batch) {
  if (!w || !batch) { set_error("bamscan_writer_write: null argument"); return BAMSCAN_ERR_INVALID; }
  if (w->finished) { set_error("bamscan_writer_write: the writer is finished"); return BAMSCAN_ERR_INVALID; }
  if (batch->n_children < w->n_cols) { set_error("bamscan_writer_write: the batch has %lld columns, the schema %d", (long long)batch->n_children, w->n_cols); return BAMSCAN_ERR_INVALID; }
  const int64_t n = batch->length;
  w->st.batches++;
  if (n == 0) return BAMSCAN_OK;
  WCU_TRY(cudaSetDevice(w->device));
  if (w->format == FMT_FASTQ) return fastq_write_impl(w, batch, n);
  auto hc = [&](int idx) { return HostCol{batch->children[idx], batch->offset + batch->children[idx]->offset}; };
  // shape checks before any buffer is touched (the arrays carry no type: the schema given at open decides how they are read)
  auto shape_ok = [&](int idx, int64_t want_buffers, bool list) {
    const ArrowArray* a = batch->children[idx];
    if (!a || !a->buffers || a->n_buffers < want_buffers || a->length + a->offset < n + batch->offset) return false;
    for (int64_t b = 1; b < want_buffers; b++) if (!a->buffers[b] && !(b == 2)) return false;     // (an all-empty Utf8 column may have no data buffer)
    if (list && (a->n_children < 1 || !a->children || !a->children[0] || !a->children[0]->buffers || a->children[0]->n_buffers < 2)) return false;
    return true;
  };
  for (int k = 0; k < 11; k++) {
    const bool utf8 = k == 0 || k == 1 || k == 4 || k == 6 || k == 8 || k == 9;
    if (!shape_ok(w->col[k], utf8 ? 3 : 2, false)) { set_error("bamscan_writer_write: column %d of the batch does not have the layout of the writer's input schema", w->col[k]); return BAMSCAN_ERR_INVALID; }
  }
  for (auto& g : w->tags)
    if (!shape_ok(g.col, g.kind == HK_Utf8 ? 3 : 2, g.kind >= HK_ListInt8 && g.kind <= HK_ListFloat32)) { set_error("bamscan_writer_write: tag column %d of the batch does not have the layout of the writer's input schema", g.col); return BAMSCAN_ERR_INVALID; }
  // ---- H2D of every buffer the encoder reads ----
  size_t need = 4096;
  if (!w->src_on_device) for (int k : {0, 1, 4, 6, 8, 9}) need += utf8_bytes(w, hc(w->col[k]), n);
  need += 5 * ((size_t)n * 4 + (size_t)n / 8 + 64);
  for (auto& g : w->tags) {
    if (w->src_on_device) break;
    const HostCol c = hc(g.col);
    if (g.kind == HK_Utf8) need += utf8_bytes(w, c, n);
    else if (g.kind >= HK_ListInt8 && g.kind <= HK_ListFloat32) {
      const int32_t* o = static_cast<const int32_t*>(c.a->buffers[1]);
      need += (size_t)(o[c.off + n] - o[c.off]) * 4 + (size_t)(n + 1) * 4 + (size_t)n / 8 + 64;
    } else need += (size_t)n * 8 + (size_t)n / 8 + 64;
  }
  int rc;
  const double t_w0 = now_ms();
  if ((rc = w->in.reserve(need))) return rc;
  enc::EncArgs A;
  memset(&A, 0, sizeof A);
  size_t cur = 0;
  if ((rc = stage_utf8(w, &cur, hc(w->col[0]), n, &A.name)) || (rc = stage_utf8(w, &cur, hc(w->col[1]), n, &A.chrom)) ||
      (rc = stage_prim(w, &cur, hc(w->col[2]), n, &A.start)) || (rc = stage_prim(w, &cur, hc(w->col[3]), n, &A.flags)) ||
      (rc = stage_utf8(w, &cur, hc(w->col[4]), n, &A.cigar)) || (rc = stage_prim(w, &cur, hc(w->col[5]), n, &A.mapq)) ||
      (rc = stage_utf8(w, &cur, hc(w->col[6]), n, &A.mate_chrom)) || (rc = stage_prim(w, &cur, hc(w->col[7]), n, &A.mate_start)) ||
      (rc = stage_utf8(w, &cur, hc(w->col[8]), n, &A.seq)) || (rc = stage_utf8(w, &cur, hc(w->col[9]), n, &A.qual)) ||
      (rc = stage_prim(w, &cur, hc(w->col[10]), n, &A.tlen)))
    return rc;
  A.n_tags = (int32_t)w->tags.size();
  for (size_t t = 0; t < w->tags.size(); t++) {
    const WTag& g = w->tags[t];
    const HostCol c = hc(g.col);
    enc::TagCol& T = A.tags[t];
    T.kind = g.kind; T.tag[0] = g.tag[0]; T.tag[1] = g.tag[1]; T.sam_type = g.sam_type; T.subtype = g.subtype; T.base = c.off;
    if (g.kind == HK_Utf8) {
      enc::Utf8Col u;
      if ((rc = stage_utf8(w, &cur, c, n, &u))) return rc;
      T.values = u.data; T.off = u.off; T.valid = u.valid;
    } else if (g.kind >= HK_ListInt8 && g.kind <= HK_ListFloat32) {
      const int32_t* o = static_cast<const int32_t*>(c.a->buffers[1]);
      uint8_t* d;
      if ((rc = stage(w, &cur, o + c.off, (size_t)(n + 1) * 4, &d))) return rc;
      T.off = reinterpret_cast<const int32_t*>(d) - c.off;
      const ArrowArray* ch = c.a->children[0];
      if (ch->null_count > 0) { set_error("SAM array tags cannot contain null elements"); return BAMSCAN_ERR_SCHEMA; }
      const size_t es = (g.kind == HK_ListInt8 || g.kind == HK_ListUInt8) ? 1 : (g.kind == HK_ListInt16 || g.kind == HK_ListUInt16) ? 2 : 4;
      int32_t first = 0, last = 0;
      if (!off_ends(w, o, c.off, c.off + n, &first, &last)) { set_error("bamscan_writer_write_device: cannot read the offsets of a device batch"); return BAMSCAN_ERR_CUDA; }
      const uint8_t* cv = static_cast<const uint8_t*>(ch->buffers[1]);
      if ((rc = stage(w, &cur, cv ? cv + (size_t)(ch->offset + first) * es : nullptr, cv ? (size_t)(last - first) * es : 0, &d))) return rc;
      T.values = d - (size_t)first * es;                   // element index = list offset (child offset already applied)
      T.child_base = 0;
      if ((rc = stage_validity(w, &cur, c, n, &T.valid))) return rc;
    } else {
      enc::PrimCol p;
      const size_t es = (g.kind == enc::WK_Int8 || g.kind == enc::WK_UInt8) ? 1 : (g.kind == enc::WK_Int16 || g.kind == enc::WK_UInt16) ? 2
                        : (g.kind == enc::WK_Int64 || g.kind == enc::WK_UInt64 || g.kind == enc::WK_Float64) ? 8 : 4;
      if ((rc = stage_prim(w, &cur, c, n, &p, es))) return rc;
      T.values = p.values; T.valid = p.valid;
    }
  }
  A.ref_blob = static_cast<const uint8_t*>(w->ref_blob.p); A.ref_off = static_cast<const int32_t*>(w->ref_off.p);
  A.ref_ids = static_cast<const int32_t*>(w->ref_ids.p); A.n_ref = w->n_ref;
  A.cigar_binary = w->cigar_binary; A.zero_based = w->zero_based;
  WTRACE("[writer] batch of %lld rows: staged %.1f MB in %.1f ms\n", (long long)n, cur / 1e6, now_ms() - t_w0);
  // ---- slices of rows: sizes -> offsets -> records -> members ----
  if ((rc = w->small.reserve(4096))) return rc;
  uint32_t* d_err = static_cast<uint32_t*>(w->small.p);
  int64_t r0 = 0;
  uint32_t want_rows = w->slice_rows;
  while (r0 < n) {
    uint32_t rows = (uint32_t)std::min<int64_t>(want_rows, n - r0);
    if ((rc = w->rec_len.reserve((size_t)rows * 4)) || (rc = w->ref_pairs.reserve((size_t)rows * 8)) || (rc = w->cig_bin.reserve((size_t)rows * 4)) ||
        (rc = w->rec_off.reserve(((size_t)rows + 1) * 8)) || (rc = w->cig_tmp.reserve((size_t)rows * 8)) || (rc = w->tile_sums.reserve(((size_t)rows / 4096 + 2) * 16)))
      return rc;
    A.row0 = (uint32_t)r0; A.n_rows = rows;
    WCU_TRY(cudaEventRecord(w->ev[0], w->stream));
    WCU_TRY(cudaMemsetAsync(d_err, 0, 16, w->stream));
    uint32_t* d_cig_ops = static_cast<uint32_t*>(w->cig_tmp.p); uint32_t* d_cig_span = d_cig_ops + rows;
    enc::enc_cigar_kernel<8><<<(((rows + 3) / 4) * 32 + 255) / 256, 256, 0, w->stream>>>(A, d_cig_ops, d_cig_span, d_err);
    enc::enc_size_kernel<<<(rows + 255) / 256, 256, 0, w->stream>>>(A, d_cig_ops, d_cig_span, static_cast<uint32_t*>(w->rec_len.p), static_cast<int32_t*>(w->ref_pairs.p),
                                                                   static_cast<uint32_t*>(w->cig_bin.p), d_err);
    w->st.kernel_launches += 2;
    uint64_t total = 0;
    const uint32_t* e = reinterpret_cast<const uint32_t*>(w->h_small + 4096);
    if ((rc = sum_lengths(w, rows, d_err, &total))) return rc;
    if (e[0]) { set_error("%s write error: row %u: %s", format_name(w->format), e[1], enc_err_text(e[0])); return enc_err_class(e[0]); }
    if (w->format == FMT_SAM) {                                // the rows passed the BAM rules: SAM line lengths + the SAM-only checks
      if (total / rows > 2048) samenc::sam_size_kernel<32><<<(rows * 32 + 255) / 256, 256, 0, w->stream>>>(A, d_cig_ops, static_cast<int32_t*>(w->ref_pairs.p), static_cast<uint32_t*>(w->rec_len.p), d_err);
      else samenc::sam_size_kernel<8><<<(((rows + 3) / 4) * 32 + 255) / 256, 256, 0, w->stream>>>(A, d_cig_ops, static_cast<int32_t*>(w->ref_pairs.p), static_cast<uint32_t*>(w->rec_len.p), d_err);
      w->st.kernel_launches += 1;
      if ((rc = sum_lengths(w, rows, d_err, &total))) return rc;
      if (e[0]) { set_error("SAM write error: row %u: %s", e[1], enc_err_text(e[0])); return enc_err_class(e[0]); }
    }
    if (total > SLICE_BYTES && rows > 1) {                   // long reads: fewer rows per pass
      want_rows = std::max<uint32_t>(1, (uint32_t)((double)rows * (double)SLICE_BYTES / (double)total * 0.9));
      w->slice_rows = want_rows;                               // (the next batch starts from this estimate)
      continue;
    }
    if ((rc = place_records(w, rows, total))) return rc;
    if (w->format == FMT_SAM) {
      const unsigned long long* d_off = static_cast<const unsigned long long*>(w->rec_off.p);
      if (total / rows > 2048) samenc::sam_records_kernel<32><<<(rows * 32 + 255) / 256, 256, 0, w->stream>>>(A, d_off, d_cig_ops, static_cast<int32_t*>(w->ref_pairs.p), static_cast<uint8_t*>(w->stream_buf.p), d_err);
      else samenc::sam_records_kernel<8><<<(((rows + 3) / 4) * 32 + 255) / 256, 256, 0, w->stream>>>(A, d_off, d_cig_ops, static_cast<int32_t*>(w->ref_pairs.p), static_cast<uint8_t*>(w->stream_buf.p), d_err);
    } else if (total / rows > 2048) {                         // long reads: a warp per row
      enc::enc_records_kernel<32><<<(rows * 32 + 255) / 256, 256, 0, w->stream>>>(A, static_cast<unsigned long long*>(w->rec_off.p), static_cast<int32_t*>(w->ref_pairs.p),
                                                                                   static_cast<uint32_t*>(w->cig_bin.p), static_cast<uint8_t*>(w->stream_buf.p), d_err);
    } else {
      const uint32_t warps = (rows + 3) / 4;
      enc::enc_records_kernel<8><<<(warps * 32 + 255) / 256, 256, 0, w->stream>>>(A, static_cast<unsigned long long*>(w->rec_off.p), static_cast<int32_t*>(w->ref_pairs.p),
                                                                                   static_cast<uint32_t*>(w->cig_bin.p), static_cast<uint8_t*>(w->stream_buf.p), d_err);
    }
    w->st.kernel_launches += 1;
    WCU_TRY(cudaEventRecord(w->ev[1], w->stream));
    WCU_TRY(cudaMemcpyAsync(w->h_small + 4096, d_err, 16, cudaMemcpyDeviceToHost, w->stream));
    WCU_TRY(cudaStreamSynchronize(w->stream));
    {
      const uint32_t* e = reinterpret_cast<const uint32_t*>(w->h_small + 4096);
      if (e[0]) { set_error("%s write error: row %u: %s", format_name(w->format), e[1], enc_err_text(e[0])); return w->format == FMT_SAM ? BAMSCAN_ERR_INVALID : BAMSCAN_ERR_SCHEMA; }
      float ms = 0; cudaEventElapsedTime(&ms, w->ev[0], w->ev[1]); w->st.ms_encode += ms; w->st.ms_total += ms;
    }
    w->st.rows += rows; w->st.bam_bytes += total;
    const double t_f0 = now_ms();
    if ((rc = writer_flush_members(w, w->pending + total, false))) return rc;
    WTRACE("[writer] slice of %u rows: encode done at +%.1f ms, members flushed in %.1f ms\n", rows, t_f0 - t_w0, now_ms() - t_f0);
    r0 += rows;
  }
  return BAMSCAN_OK;
}

// Appends `bytes` device bytes to the file: D2H into a free pinned staging buffer, then its pieces go to the file threads.
// Returns once every D2H has landed (the device bytes may be overwritten then).
static int writer_emit(BamWriter* w, const uint8_t* dev, uint64_t bytes) {
  for (uint64_t at = 0; at < bytes; at += OUT_CHUNK) {
    const size_t nb = (size_t)std::min<uint64_t>(OUT_CHUNK, bytes - at);
    int slot = -1;
    {
      std::unique_lock<std::mutex> lk(w->mu);
      w->cv.wait(lk, [&] { for (int b = 0; b < OUT_BUFS; b++) if (!w->out_busy[b]) { slot = b; return true; } return w->file_failed; });
      if (w->file_failed || slot < 0) { set_error("Failed to write %s record: write(%s) failed", format_name(w->format), w->path.c_str()); return BAMSCAN_ERR_IO; }
      w->out_busy[slot] = FILE_THREADS;
    }
    WCU_TRY(cudaMemcpyAsync(w->h_out[slot], dev + at, nb, cudaMemcpyDeviceToHost, w->stream));
    WCU_TRY(cudaStreamSynchronize(w->stream));
    {
      std::lock_guard<std::mutex> lk(w->mu);
      const size_t per = (nb + FILE_THREADS - 1) / FILE_THREADS;
      for (int t = 0; t < FILE_THREADS; t++) {
        const size_t b = std::min(nb, per * t), e = std::min(nb, b + per);
        w->file_q.push_back(BamWriter::FileJob{slot, b, e - b, w->file_off + b});
      }
      w->file_off += nb;
    }
    w->cv.notify_all();
  }
  WCU_TRY(cudaStreamSynchronize(w->stream));
  return BAMSCAN_OK;
}

// Compresses the full members of the first `total` bytes of the stream buffer (all of them when final_flush) and appends them
// to the file; the remaining tail moves to the front of the buffer.  Plain (FASTQ compression 2): the bytes go to the file as
// they are, nothing stays behind.
static int writer_flush_members(BamWriter* w, uint64_t total, bool final_flush) {
  if (w->plain) {
    int rc;
    if (total && (rc = writer_emit(w, static_cast<const uint8_t*>(w->stream_buf.p), total))) return rc;
    w->st.compressed_bytes += total;
    w->pending = 0;
    return BAMSCAN_OK;
  }
  const uint64_t n_members = final_flush ? (total + dfl::BLOCK - 1) / dfl::BLOCK : total / dfl::BLOCK;
  if (n_members == 0) { w->pending = total; return BAMSCAN_OK; }
  const uint64_t consumed = std::min<uint64_t>(total, n_members * dfl::BLOCK);
  int rc;
  const uint32_t grid = (uint32_t)std::min<uint64_t>(n_members, 2ull * w->n_sms);
  if ((rc = w->slots.reserve(n_members * dfl::SLOT)) || (rc = w->sizes.reserve(n_members * 4)) || (rc = w->offsets.reserve(n_members * 8 + 16)) ||
      (rc = w->tok.reserve((size_t)grid * dfl::SLOT * 4)))
    return rc;
  uint32_t* d_ticket = static_cast<uint32_t*>(w->small.p) + 8;
  unsigned long long* d_total = reinterpret_cast<unsigned long long*>(static_cast<uint32_t*>(w->small.p) + 16);
  WCU_TRY(cudaEventRecord(w->ev[2], w->stream));
  WCU_TRY(cudaMemsetAsync(d_ticket, 0, 4, w->stream));
  dfl::bgzf_deflate_kernel<<<grid, dfl::NT, sizeof(dfl::Smem), w->stream>>>(static_cast<const uint8_t*>(w->stream_buf.p), consumed, (uint32_t)n_members,
                                                                           static_cast<uint8_t*>(w->slots.p), static_cast<uint32_t*>(w->sizes.p),
                                                                           static_cast<uint32_t*>(w->tok.p), d_ticket, w->compression == 1);
  cta_scan_kernel<<<1, CTA_SCAN_THREADS, 0, w->stream>>>(static_cast<const uint32_t*>(w->sizes.p), static_cast<unsigned long long*>(w->offsets.p), (uint32_t)n_members, d_total);
  WCU_TRY(cudaEventRecord(w->ev[3], w->stream));
  WCU_TRY(cudaMemcpyAsync(w->h_small + 5000, d_total, 8, cudaMemcpyDeviceToHost, w->stream));
  WCU_TRY(cudaStreamSynchronize(w->stream));
  WCU_TRY(cudaGetLastError());
  const uint64_t packed_bytes = w->h_small[5000];
  const double t_d = now_ms();
  if ((rc = w->packed.reserve(packed_bytes + 16))) return rc;
  WCU_TRY(cudaEventRecord(w->ev2[0], w->stream));
  dfl::bgzf_gather_kernel<<<(uint32_t)n_members, 256, 0, w->stream>>>(static_cast<const uint8_t*>(w->slots.p), static_cast<uint32_t*>(w->sizes.p),
                                                                     static_cast<unsigned long long*>(w->offsets.p), static_cast<uint8_t*>(w->packed.p));
  WCU_TRY(cudaEventRecord(w->ev2[1], w->stream));
  w->st.kernel_launches += 3;
  // the tail moves to the front (source and destination cannot overlap: the tail is shorter than one member)
  const uint64_t tail = total - consumed;
  if (tail) WCU_TRY(cudaMemcpyAsync(w->stream_buf.p, static_cast<uint8_t*>(w->stream_buf.p) + consumed, tail, cudaMemcpyDeviceToDevice, w->stream));
  if ((rc = writer_emit(w, static_cast<const uint8_t*>(w->packed.p), packed_bytes))) return rc;
  WTRACE("[writer] %llu members, %.1f MB packed: gather + D2H + queueing %.1f ms\n", (unsigned long long)n_members, packed_bytes / 1e6, now_ms() - t_d);
  { float ms = 0, ms2 = 0; cudaEventElapsedTime(&ms, w->ev[2], w->ev[3]); cudaEventElapsedTime(&ms2, w->ev2[0], w->ev2[1]); w->st.ms_deflate += ms + ms2; w->st.ms_total += ms + ms2; }
  w->st.members += n_members; w->st.compressed_bytes += packed_bytes;
  w->pending = tail;
  return BAMSCAN_OK;
}

static int writer_finish_impl(BamWriter* w, uint64_t* rows_written) {
  if (!w) { set_error("bamscan_writer_finish: null argument"); return BAMSCAN_ERR_INVALID; }
  const double t_fin = now_ms();
  if (!w->finished) {
    WCU_TRY(cudaSetDevice(w->device));
    int rc;
    if ((rc = w->small.reserve(4096))) return rc;
    if ((rc = writer_flush_members(w, w->pending, true))) return rc;
    {
      std::unique_lock<std::mutex> lk(w->mu);
      w->cv.wait(lk, [&] { if (!w->file_q.empty()) return false; for (int b = 0; b < OUT_BUFS; b++) if (w->out_busy[b]) return false; return true; });
      if (w->file_failed) { set_error("Failed to finish %s stream: write(%s) failed", format_name(w->format), w->path.c_str()); return BAMSCAN_ERR_IO; }
    }
    if (!w->plain) {
      static const uint8_t eof_marker[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
      if (::pwrite(w->fd, eof_marker, 28, (off_t)w->file_off) != 28) { set_error("Failed to finish %s stream: write(%s) failed", format_name(w->format), w->path.c_str()); return BAMSCAN_ERR_IO; }
      w->st.compressed_bytes += 28;
    }
    ::close(w->fd); w->fd = -1;
    w->finished = true;
    WTRACE("[writer] finish: %.1f ms\n", now_ms() - t_fin);
  }
  if (rows_written) *rows_written = w->st.rows;
  return BAMSCAN_OK;
}

}  // namespace bamscan

extern "C" {

#define WRITER_GUARD(call)                                                                                           \
  try { return (call); }                                                                                             \
  catch (const std::bad_alloc&) { set_error("out of memory"); return BAMSCAN_ERR_INVALID; }                          \
  catch (const std::exception& e) { set_error("internal error: %s", e.what()); return BAMSCAN_ERR_INVALID; }          \
  catch (...) { set_error("internal error"); return BAMSCAN_ERR_INVALID; }

int bamscan_writer_open(const char* output_path, const char* sam_header_text, int32_t n_ref, const char* const* ref_names,
                        const int32_t* ref_lengths, const struct ArrowSchema* input_schema, const BamWriteOptions* options, BamWriter** out) {
  WRITER_GUARD(writer_open_impl(output_path, sam_header_text, n_ref, ref_names, ref_lengths, input_schema, options, out))
}
int bamscan_fastq_writer_open(const char* output_path, const struct ArrowSchema* input_schema, const BamWriteOptions* options, BamWriter** out) {
  WRITER_GUARD(fastq_writer_open_impl(output_path, input_schema, options, out))
}
int bamscan_sam_writer_open(const char* output_path, const char* sam_header_text, int32_t n_ref, const char* const* ref_names,
                            const int32_t* ref_lengths, const struct ArrowSchema* input_schema, const BamWriteOptions* options, BamWriter** out) {
  WRITER_GUARD(writer_open_impl(output_path, sam_header_text, n_ref, ref_names, ref_lengths, input_schema, options, out, FMT_SAM))
}
int bamscan_writer_write(BamWriter* w, const struct ArrowArray* batch) { WRITER_GUARD(writer_write_impl(w, batch)) }
static int writer_write_device_impl(BamWriter* w, const struct ArrowDeviceArray* batch) {
  if (!w || !batch) { set_error("bamscan_writer_write_device: null argument"); return BAMSCAN_ERR_INVALID; }
  if (batch->device_type != ARROW_DEVICE_CUDA || batch->device_id != w->device) { set_error("bamscan_writer_write_device: the batch lives on device %lld (type %d), the writer on CUDA device %d", (long long)batch->device_id, (int)batch->device_type, w->device); return BAMSCAN_ERR_INVALID; }
  if (cudaSetDevice(w->device) != cudaSuccess) { set_error("cudaSetDevice(%d) failed", w->device); return BAMSCAN_ERR_CUDA; }
  if (batch->sync_event && cudaStreamWaitEvent(w->stream, *static_cast<cudaEvent_t*>(batch->sync_event), 0) != cudaSuccess) { set_error("cudaStreamWaitEvent on the batch's sync_event failed"); return BAMSCAN_ERR_CUDA; }
  if (batch->sync_event && cudaEventSynchronize(*static_cast<cudaEvent_t*>(batch->sync_event)) != cudaSuccess) { set_error("waiting for the batch's sync_event failed"); return BAMSCAN_ERR_CUDA; }   // (offset ends are read with plain cudaMemcpy)
  w->src_on_device = true;
  const int rc = writer_write_impl(w, &batch->array);
  w->src_on_device = false;
  return rc;
}
int bamscan_writer_write_device(BamWriter* w, const struct ArrowDeviceArray* batch) { WRITER_GUARD(writer_write_device_impl(w, batch)) }
int bamscan_writer_finish(BamWriter* w, uint64_t* rows_written) { WRITER_GUARD(writer_finish_impl(w, rows_written)) }
int bamscan_writer_stats(const BamWriter* w, BamWriteStats* out) {
  if (!w || !out) { set_error("bamscan_writer_stats: null argument"); return BAMSCAN_ERR_INVALID; }
  *out = w->st;
  return BAMSCAN_OK;
}
void bamscan_writer_free(BamWriter* w) {
  if (!w) return;
  cudaSetDevice(w->device);
  if (w->stream) cudaStreamSynchronize(w->stream);
  { std::lock_guard<std::mutex> lk(w->mu); w->file_stop = true; }
  w->cv.notify_all();
  for (auto& th : w->file_thread) if (th.joinable()) th.join();
  if (w->fd >= 0) ::close(w->fd);
  {
    std::lock_guard<std::mutex> lk(g_res_mu);
    WriterRes& pooled = g_res_pool[w->device & 63];
    if (w->ready && !pooled.ready) { pooled = static_cast<WriterRes&>(*w); static_cast<WriterRes&>(*w) = WriterRes(); }
  }
  w->destroy();
  delete w;
}

}  // extern "C"
