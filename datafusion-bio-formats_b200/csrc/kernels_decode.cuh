// kernels_decode.cuh -- projected columnar decode of BAM records into Arrow buffers.
//
// Replaces the per-record extraction block + Arrow builders of the reference:
//   datafusion/bio-format-bam/src/physical_exec.rs:412-540   (12 guarded column appends + tags)
//   datafusion/bio-format-core/src/alignment_utils.rs:459-643,667-701 (builders, CIGAR text)
//   datafusion/bio-format-core/src/sam_tag_io.rs:154-204,658-1036 (tag walk + coercions)
//
// Three phases per chunk, all driven by rec_off[] (kernels_boundary.cuh):
//   decode_fixed_kernel  : one THREAD per record.  Fixed-width columns, validity bitmaps (warp ballots),
//                          per-row byte lengths of every projected var-len column, one aux walk that
//                          locates / converts every requested tag.
//   multi_scan_*         : exclusive prefix sums turning the length arrays into Arrow i32 offsets
//                          (all var-len columns in one launch, grid.y = column).
//   decode_var_kernel    : a group of 8 lanes (short reads) or a whole warp (long reads) per record.  Copies / transcodes the var-len payloads to their final
//                          offsets: name, chrom / mate_chrom (dictionary expand), CIGAR text (or raw words),
//                          sequence (4-bit -> ASCII via shared LUT), qualities (+33), Z/H/A/int-as-text tags,
//                          B arrays with element-wise checked conversion.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "f32_text.h"

#include "kernels_boundary.cuh"

namespace bamscan {

constexpr int MAX_TAGS = 32;        // projected tag columns per scan (DecodeParams travels as a kernel argument: 48 B per tag)

enum ColKind : int32_t {
  K_Int32 = 1, K_UInt32 = 2, K_Float32 = 3, K_Utf8 = 4, K_Binary = 5,
  K_ListInt8 = 10, K_ListUInt8 = 11, K_ListInt16 = 12, K_ListUInt16 = 13, K_ListInt32 = 14, K_ListUInt32 = 15, K_ListFloat32 = 16
};

enum DecodeErr : uint32_t {
  DEC_OK = 0, DEC_ERR_FIELDS = 1 /* record fields exceed block_size */, DEC_ERR_REF = 2 /* reference id out of range */,
  DEC_ERR_CIGAR_OP = 3, DEC_ERR_TAG_RANGE = 4 /* value does not fit the column type */, DEC_ERR_TAG_TYPE = 5 /* value kind vs column kind */,
  DEC_ERR_UNSUPPORTED_F2S = 6 /* (retired: float tags are rendered into Utf8 columns, f32_text.h) */, DEC_ERR_QUAL = 7 /* quality in 95..222: char::from(q + 33) is a two-byte UTF-8 sequence (unpinned; 0xFF wraps to ' ' and is fine) */,
  DEC_ERR_NAME = 8 /* non-ASCII read name (unpinned) */
};

struct TagPlan {
  uint32_t* valid;    // validity bitmap words
  uint32_t* values;   // fixed-width values (Int32 / UInt32 / Float32)
  int32_t* lens;      // Utf8 / List: per-row byte (Utf8) or element (List) counts -> offsets after the scan [n+1]
  uint32_t* src;      // Utf8 / List: offset in U of the aux field's TYPE byte (0 = null)
  uint8_t* data;      // Utf8 bytes / list child values
  int32_t kind;
  uint16_t tag;       // two tag bytes, little endian
  uint16_t pad;
};

struct DecodeParams {
  const uint8_t* U;
  const uint32_t* rec_off;
  uint32_t n;
  int32_t zero_based, binary_cigar, n_ref, n_tags;
  const uint32_t* ref_name_off;   // [n_ref + 1] offsets into ref_names
  const uint8_t* ref_names;
  uint32_t *start, *end, *flags, *mapq, *mate_start;
  int32_t* tlen;
  uint32_t *v_chrom, *v_start, *v_end, *v_mchrom, *v_mstart;
  int32_t *l_name, *l_chrom, *l_cigar, *l_mchrom, *l_seq, *l_qual;
  uint8_t *d_name, *d_chrom, *d_cigar, *d_mchrom, *d_seq, *d_qual;
  uint32_t* err;                  // [0] code, [1] row
  // SAM handles only (kernels_sam.cuh); 0 / null on BAM handles, whose results these leave unchanged.  noodles-sam's RecordBuf
  // differs from the lazy BAM record in two places:
  int32_t end_zero_span;          // 1: a placed read whose CIGAR spans no reference base has end = start + 0 - 1 (1-based), not NULL;
                                  // NULL again at POS 1, where that is 0 (RecordBuf::alignment_end goes through Position::new)
  const uint8_t* qual_absent;     // [n]: 1 = QUAL was '*' with a non-empty SEQ: the quality string is empty, not 0xFF fill
  TagPlan tags[MAX_TAGS];
};

__device__ __forceinline__ void set_err(uint32_t* err, uint32_t code, uint32_t row) {
  if (atomicCAS(&err[0], 0u, code) == 0u) err[1] = row;
}

__device__ __forceinline__ uint32_t ndigits_u32(uint32_t v) {
  return v < 10u ? 1u : v < 100u ? 2u : v < 1000u ? 3u : v < 10000u ? 4u : v < 100000u ? 5u : v < 1000000u ? 6u :
         v < 10000000u ? 7u : v < 100000000u ? 8u : v < 1000000000u ? 9u : 10u;
}
__device__ __forceinline__ bool is_scalar_value(int64_t v) { return v >= 0 && v <= 0x10FFFF && !(v >= 0xD800 && v <= 0xDFFF); }
__device__ __forceinline__ uint32_t utf8_len(uint32_t cp) { return cp < 0x80u ? 1u : cp < 0x800u ? 2u : cp < 0x10000u ? 3u : 4u; }
__device__ __forceinline__ uint32_t sub_size(uint8_t st) {
  return (st == 'c' || st == 'C') ? 1u : (st == 's' || st == 'S') ? 2u : (st == 'i' || st == 'I' || st == 'f') ? 4u : 0u;
}

// strict UTF-8 validation of U[o .. o+n)
__device__ __forceinline__ bool utf8_valid(const uint8_t* U, uint32_t o, uint32_t n) {
  uint32_t i = 0;
  while (i < n) {
    uint32_t c = U[o + i];
    if (c < 0x80u) { i++; continue; }
    uint32_t len, cp;
    if ((c & 0xE0u) == 0xC0u) { len = 2; cp = c & 0x1Fu; }
    else if ((c & 0xF0u) == 0xE0u) { len = 3; cp = c & 0x0Fu; }
    else if ((c & 0xF8u) == 0xF0u) { len = 4; cp = c & 0x07u; }
    else return false;
    if (i + len > n) return false;
    for (uint32_t k = 1; k < len; k++) { uint32_t d = U[o + i + k]; if ((d & 0xC0u) != 0x80u) return false; cp = (cp << 6) | (d & 0x3Fu); }
    if ((len == 2 && cp < 0x80u) || (len == 3 && cp < 0x800u) || (len == 4 && cp < 0x10000u)) return false;
    if (cp > 0x10FFFFu || (cp >= 0xD800u && cp <= 0xDFFFu)) return false;
    i += len;
  }
  return true;
}

// One aux field -> the requested column's representation (sam_tag_io.rs:658-741 scalars, :761-1036 arrays are sized here and
// converted in decode_var_kernel).  `a` = offset of the field's tag bytes, `v` = offset of its value, vlen = value bytes.
struct TagConv { bool ok; uint32_t val; int32_t len; uint32_t src; };
__device__ __forceinline__ TagConv convert_tag(const DecodeParams& P, const TagPlan& T, const uint8_t* U, uint32_t a, uint8_t ty, uint32_t v,
                                               uint32_t vlen, bool utf8_ok, uint32_t r) {
  const int32_t kind = T.kind;
  bool ok = true; uint32_t val = 0; int32_t len = 0; uint32_t src = 0;
  int64_t iv = 0; bool is_int = true;
  switch (ty) {
    case 'c': iv = (int8_t)U[v]; break;
    case 'C': iv = U[v]; break;
    case 's': iv = (int16_t)ld_u16(U, v); break;
    case 'S': iv = ld_u16(U, v); break;
    case 'i': iv = (int32_t)ld_u32(U, v); break;
    case 'I': iv = ld_u32(U, v); break;
    default: is_int = false; break;
  }
  if (is_int) {
    if (kind == K_Int32) { if (iv < -2147483648ll || iv > 2147483647ll) { set_err(P.err, DEC_ERR_TAG_RANGE, r); ok = false; } val = (uint32_t)(int32_t)iv; }
    else if (kind == K_UInt32) { if (iv < 0) { set_err(P.err, DEC_ERR_TAG_RANGE, r); ok = false; } val = (uint32_t)iv; }
    else if (kind == K_Utf8) { len = is_scalar_value(iv) ? (int32_t)utf8_len((uint32_t)iv) : (int32_t)(ndigits_u32((uint32_t)(iv < 0 ? -iv : iv)) + (iv < 0 ? 1u : 0u)); src = a + 2u; }
    else { set_err(P.err, DEC_ERR_TAG_TYPE, r); ok = false; }
  } else if (ty == 'f') {
    if (kind == K_Float32) val = ld_u32(U, v);
    else if (kind == K_Utf8) { len = (int32_t)f32_to_text(ld_u32(U, v), nullptr); src = a + 2u; }     // f32::to_string() (sam_tag_io.rs:670-676)
    else { set_err(P.err, DEC_ERR_TAG_TYPE, r); ok = false; }
  } else if (ty == 'A') {
    if (kind == K_Int32 || kind == K_UInt32) val = U[v];
    else if (kind == K_Utf8) { len = U[v] < 0x80 ? 1 : 2; src = a + 2u; }
    else { set_err(P.err, DEC_ERR_TAG_TYPE, r); ok = false; }
  } else if (ty == 'Z' || ty == 'H') {
    if (kind == K_Utf8) { if (utf8_ok) { len = (int32_t)(vlen - 1u); src = a + 2u; } else ok = false; /* invalid UTF-8 -> NULL */ }
    else { set_err(P.err, DEC_ERR_TAG_TYPE, r); ok = false; }
  } else {   // 'B'
    uint8_t st = U[v];
    if (kind >= K_ListInt8 && !(st == 'f' && kind != K_ListFloat32)) { len = (int32_t)ld_u32(U, v + 1); src = a + 2u; }
    else { set_err(P.err, DEC_ERR_TAG_TYPE, r); ok = false; }
  }
  TagConv c; c.ok = ok; c.val = ok ? val : 0u; c.len = ok ? len : 0; c.src = ok ? src : 0u;
  return c;
}

// ---------------------------------------------------------------------------------------------
// phase 1: one thread per record
__global__ void __launch_bounds__(256, 4)
decode_fixed_kernel(const DecodeParams P) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool act = r < P.n;
  const uint8_t* U = P.U;
  uint32_t o = 0, bs = 32;
  int32_t ref = -1, pos = -1, nref = -1, npos = -1, tlen = 0, l_seq = 0;
  uint32_t l_name = 1, mapq = 0, n_cig = 0, flag = 0;
  if (act) {
    o = P.rec_off[r];
    bs = ld_u32(U, o);
    ref = (int32_t)ld_u32(U, o + 4); pos = (int32_t)ld_u32(U, o + 8);
    uint32_t w = ld_u32(U, o + 12); l_name = w & 0xffu; mapq = (w >> 8) & 0xffu;
    w = ld_u32(U, o + 16); n_cig = w & 0xffffu; flag = w >> 16;
    l_seq = (int32_t)ld_u32(U, o + 20);
    nref = (int32_t)ld_u32(U, o + 24); npos = (int32_t)ld_u32(U, o + 28); tlen = (int32_t)ld_u32(U, o + 32);
  }
  const uint32_t o_name = o + 36, o_cig = o_name + l_name, o_seq = o_cig + 4u * n_cig;
  const uint32_t o_qual = o_seq + ((uint32_t)l_seq + 1u) / 2u, o_aux = o_qual + (uint32_t)l_seq, o_end = o + 4u + bs;
  if (act) {
    uint64_t need = 32ull + l_name + 4ull * n_cig + ((uint64_t)(uint32_t)l_seq + 1) / 2 + (uint64_t)(uint32_t)l_seq;
    if (l_seq < 0 || need > bs) set_err(P.err, DEC_ERR_FIELDS, r);
    if (ref < -1 || ref >= P.n_ref || nref < -1 || nref >= P.n_ref) set_err(P.err, DEC_ERR_REF, r);
  }
  const bool sane = act && l_seq >= 0 && (uint64_t)(o_aux - o - 4u) <= bs && ref >= -1 && ref < P.n_ref && nref >= -1 && nref < P.n_ref;

  // CIGAR walk: reference span (M/D/N/=/X) and rendered text length
  uint32_t span = 0, cig_txt = 0;
  if (sane && (P.end || (P.l_cigar && !P.binary_cigar))) {
    for (uint32_t k = 0; k < n_cig; k++) {
      uint32_t w = ld_u32(U, o_cig + 4u * k), op = w & 15u, len = w >> 4;
      if (op > 8u) { set_err(P.err, DEC_ERR_CIGAR_OP, r); break; }
      if ((0x18Du >> op) & 1u) span += len;          // ops 0,2,3,7,8
      cig_txt += ndigits_u32(len) + 1u;
    }
  }
  const bool has_start = sane && pos >= 0;
  const bool has_end = has_start && (span > 0 || (P.end_zero_span && pos > 0));     // noodles bam::Record::alignment_end: None when the span is 0
  const bool has_mstart = sane && npos >= 0;
  if (act) {
    if (P.start) P.start[r] = has_start ? (uint32_t)pos + (P.zero_based ? 0u : 1u) : 0u;
    if (P.end) P.end[r] = has_end ? (uint32_t)pos + span : 0u;                 // 1-based inclusive end == 0-based exclusive end
    if (P.flags) P.flags[r] = flag;
    if (P.mapq) P.mapq[r] = mapq;
    if (P.mate_start) P.mate_start[r] = has_mstart ? (uint32_t)npos + (P.zero_based ? 0u : 1u) : 0u;
    if (P.tlen) P.tlen[r] = tlen;
    if (P.l_name) P.l_name[r] = sane ? (int32_t)(l_name ? l_name - 1u : 0u) : 0;
    if (P.l_chrom) P.l_chrom[r] = (sane && ref >= 0) ? (int32_t)(P.ref_name_off[ref + 1] - P.ref_name_off[ref]) : 0;
    if (P.l_mchrom) P.l_mchrom[r] = (sane && nref >= 0) ? (int32_t)(P.ref_name_off[nref + 1] - P.ref_name_off[nref]) : 0;
    if (P.l_cigar) P.l_cigar[r] = sane ? (int32_t)(P.binary_cigar ? 4u * n_cig : cig_txt) : 0;
    if (P.l_seq) P.l_seq[r] = sane ? l_seq : 0;
    if (P.l_qual) P.l_qual[r] = (sane && !(P.qual_absent && P.qual_absent[r])) ? l_seq : 0;
  }
  // validity bitmaps: one 32-bit word per warp (rows are warp aligned)
  uint32_t m;
  if (P.v_chrom) { m = __ballot_sync(0xffffffffu, sane && ref >= 0); if (lane == 0 && act) P.v_chrom[r >> 5] = m; }
  if (P.v_start) { m = __ballot_sync(0xffffffffu, has_start); if (lane == 0 && act) P.v_start[r >> 5] = m; }
  if (P.v_end) { m = __ballot_sync(0xffffffffu, has_end); if (lane == 0 && act) P.v_end[r >> 5] = m; }
  if (P.v_mchrom) { m = __ballot_sync(0xffffffffu, sane && nref >= 0); if (lane == 0 && act) P.v_mchrom[r >> 5] = m; }
  if (P.v_mstart) { m = __ballot_sync(0xffffffffu, has_mstart); if (lane == 0 && act) P.v_mstart[r >> 5] = m; }

  if (P.n_tags == 0) return;
  // ---- aux walk (sam_tag_io.rs:154-204): every field is visited once, requested tags are converted in place
  uint32_t valid_mask = 0, seen = 0;
  if (sane) {
    uint32_t a = o_aux;
    while (a + 3u <= o_end) {
      uint32_t tag = ld_u16(U, a); uint8_t ty = U[a + 2];
      uint32_t v = a + 3u, rem = o_end - v, vlen;
      if (ty == 'A' || ty == 'c' || ty == 'C') vlen = 1;
      else if (ty == 's' || ty == 'S') vlen = 2;
      else if (ty == 'i' || ty == 'I' || ty == 'f') vlen = 4;
      else if (ty == 'Z' || ty == 'H') { uint32_t k = 0; while (k < rem && U[v + k] != 0) k++; if (k >= rem) break; vlen = k + 1u; }
      else if (ty == 'B') { if (rem < 5u) break; uint32_t es = sub_size(U[v]); if (!es) break; uint64_t need = 5ull + (uint64_t)ld_u32(U, v + 1) * es; if (need > rem) break; vlen = (uint32_t)need; }
      else break;                                   // malformed field: the reference warns and stops yielding fields
      if (vlen > rem) break;
      int t = -1;
      for (int k = 0; k < P.n_tags; k++) if (P.tags[k].tag == tag) t = k;   // HashMap<Tag, idx>: the last duplicate name wins
      if (t >= 0) {
        const TagPlan& T = P.tags[t];
        const bool utf8_ok = (T.kind == K_Utf8 && (ty == 'Z' || ty == 'H')) ? utf8_valid(U, v, vlen - 1u) : true;
        const TagConv c = convert_tag(P, T, U, a, ty, v, vlen, utf8_ok, r);
        seen |= 1u << t;
        if (c.ok) valid_mask |= 1u << t; else valid_mask &= ~(1u << t);
        if (T.values) T.values[r] = c.val;
        if (T.lens) T.lens[r] = c.len;
        if (T.src) T.src[r] = c.src;
      }
      a = v + vlen;
    }
  }
  for (int t = 0; t < P.n_tags; t++) {
    const TagPlan& T = P.tags[t];
    if (T.valid) { m = __ballot_sync(0xffffffffu, (valid_mask >> t) & 1u); if (lane == 0 && act) T.valid[r >> 5] = m; }
    if (act && !((seen >> t) & 1u)) {
      if (T.values) T.values[r] = 0u;
      if (T.lens) T.lens[r] = 0;
      if (T.src) T.src[r] = 0u;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// phase 1 for LONG records (mean record > 2 KiB: long-read BAMs): one warp per row, the lanes co-operate inside the
// record -- CIGAR ops are strided over the lanes, Z/H strings are measured and ASCII-checked 32 bytes at a time.  Same
// results as decode_fixed_kernel; validity bits are OR-ed into the (pre-zeroed) bitmap words.
__global__ void __launch_bounds__(256)
decode_fixed_warp_kernel(const DecodeParams P) {
  const int lane = threadIdx.x & 31;
  const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= P.n) return;
  const uint8_t* U = P.U;
  {
    const uint32_t o = P.rec_off[r];
    const uint32_t bs = ld_u32(U, o);
    const int32_t ref = (int32_t)ld_u32(U, o + 4), pos = (int32_t)ld_u32(U, o + 8);
    uint32_t x = ld_u32(U, o + 12); const uint32_t l_name = x & 0xffu, mapq = (x >> 8) & 0xffu;
    x = ld_u32(U, o + 16); const uint32_t n_cig = x & 0xffffu, flag = x >> 16;
    const int32_t l_seq = (int32_t)ld_u32(U, o + 20);
    const int32_t nref = (int32_t)ld_u32(U, o + 24), npos = (int32_t)ld_u32(U, o + 28), tlen = (int32_t)ld_u32(U, o + 32);
    const uint32_t o_name = o + 36, o_cig = o_name + l_name, o_seq = o_cig + 4u * n_cig;
    const uint32_t o_qual = o_seq + ((uint32_t)l_seq + 1u) / 2u, o_aux = o_qual + (uint32_t)l_seq, o_end = o + 4u + bs;
    const uint64_t need = 32ull + l_name + 4ull * n_cig + ((uint64_t)(uint32_t)l_seq + 1) / 2 + (uint64_t)(uint32_t)l_seq;
    if (lane == 0) {
      if (l_seq < 0 || need > bs) set_err(P.err, DEC_ERR_FIELDS, r);
      if (ref < -1 || ref >= P.n_ref || nref < -1 || nref >= P.n_ref) set_err(P.err, DEC_ERR_REF, r);
    }
    const bool sane = l_seq >= 0 && need <= bs && ref >= -1 && ref < P.n_ref && nref >= -1 && nref < P.n_ref;
    uint32_t span = 0, cig_txt = 0;
    if (sane && (P.end || (P.l_cigar && !P.binary_cigar))) {
      bool bad_op = false;
      for (uint32_t k = lane; k < n_cig; k += 32) {
        uint32_t cw = ld_u32(U, o_cig + 4u * k), op = cw & 15u, len = cw >> 4;
        bad_op |= op > 8u;
        if ((0x18Du >> op) & 1u) span += len;
        cig_txt += ndigits_u32(len) + 1u;
      }
      #pragma unroll
      for (int s2 = 16; s2; s2 >>= 1) { span += __shfl_xor_sync(0xffffffffu, span, s2); cig_txt += __shfl_xor_sync(0xffffffffu, cig_txt, s2); }
      if (__any_sync(0xffffffffu, bad_op) && lane == 0) set_err(P.err, DEC_ERR_CIGAR_OP, r);
    }
    const bool has_start = sane && pos >= 0, has_end = has_start && (span > 0 || (P.end_zero_span && pos > 0)), has_mstart = sane && npos >= 0;
    if (lane == 0) {
      if (P.start) P.start[r] = has_start ? (uint32_t)pos + (P.zero_based ? 0u : 1u) : 0u;
      if (P.end) P.end[r] = has_end ? (uint32_t)pos + span : 0u;
      if (P.flags) P.flags[r] = flag;
      if (P.mapq) P.mapq[r] = mapq;
      if (P.mate_start) P.mate_start[r] = has_mstart ? (uint32_t)npos + (P.zero_based ? 0u : 1u) : 0u;
      if (P.tlen) P.tlen[r] = tlen;
      if (P.l_name) P.l_name[r] = sane ? (int32_t)(l_name ? l_name - 1u : 0u) : 0;
      if (P.l_chrom) P.l_chrom[r] = (sane && ref >= 0) ? (int32_t)(P.ref_name_off[ref + 1] - P.ref_name_off[ref]) : 0;
      if (P.l_mchrom) P.l_mchrom[r] = (sane && nref >= 0) ? (int32_t)(P.ref_name_off[nref + 1] - P.ref_name_off[nref]) : 0;
      if (P.l_cigar) P.l_cigar[r] = sane ? (int32_t)(P.binary_cigar ? 4u * n_cig : cig_txt) : 0;
      if (P.l_seq) P.l_seq[r] = sane ? l_seq : 0;
      if (P.l_qual) P.l_qual[r] = (sane && !(P.qual_absent && P.qual_absent[r])) ? l_seq : 0;
    }
    const uint32_t bit = 1u << (r & 31u), word = r >> 5;
    if (lane == 0) {
      if (P.v_chrom && sane && ref >= 0) atomicOr(&P.v_chrom[word], bit);
      if (P.v_start && has_start) atomicOr(&P.v_start[word], bit);
      if (P.v_end && has_end) atomicOr(&P.v_end[word], bit);
      if (P.v_mchrom && sane && nref >= 0) atomicOr(&P.v_mchrom[word], bit);
      if (P.v_mstart && has_mstart) atomicOr(&P.v_mstart[word], bit);
    }
    if (P.n_tags == 0) return;
    uint32_t valid_mask = 0, seen = 0;
    if (sane) {
      uint32_t a = o_aux;
      while (a + 3u <= o_end) {
        const uint32_t tag = ld_u16(U, a); const uint8_t ty = U[a + 2];
        const uint32_t v = a + 3u, rem = o_end - v;
        uint32_t vlen; bool ascii = true;
        if (ty == 'A' || ty == 'c' || ty == 'C') vlen = 1;
        else if (ty == 's' || ty == 'S') vlen = 2;
        else if (ty == 'i' || ty == 'I' || ty == 'f') vlen = 4;
        else if (ty == 'Z' || ty == 'H') {
          uint32_t found = 0xffffffffu;
          for (uint32_t b0 = 0; b0 < rem && found == 0xffffffffu; b0 += 32) {    // uniform trip count
            const uint32_t k = b0 + lane;
            const uint8_t c = k < rem ? U[v + k] : (uint8_t)1;
            const uint32_t z = __ballot_sync(0xffffffffu, k < rem && c == 0);
            const uint32_t hi = __ballot_sync(0xffffffffu, k < rem && c >= 0x80);
            if (z) { found = b0 + (uint32_t)__ffs(z) - 1u; ascii &= (hi & ((1u << (__ffs(z) - 1)) - 1u)) == 0u; }
            else ascii &= hi == 0u;
          }
          if (found == 0xffffffffu) break;
          vlen = found + 1u;
        }
        else if (ty == 'B') { if (rem < 5u) break; uint32_t es = sub_size(U[v]); if (!es) break; uint64_t nb2 = 5ull + (uint64_t)ld_u32(U, v + 1) * es; if (nb2 > rem) break; vlen = (uint32_t)nb2; }
        else break;
        if (vlen > rem) break;
        int t = -1;
        for (int k = 0; k < P.n_tags; k++) if (P.tags[k].tag == tag) t = k;
        if (t >= 0) {
          const TagPlan& T = P.tags[t];
          const bool utf8_ok = (T.kind == K_Utf8 && (ty == 'Z' || ty == 'H') && !ascii) ? utf8_valid(U, v, vlen - 1u) : true;
          const TagConv c = convert_tag(P, T, U, a, ty, v, vlen, utf8_ok, r);
          seen |= 1u << t;
          if (c.ok) valid_mask |= 1u << t; else valid_mask &= ~(1u << t);
          if (lane == 0) {
            if (T.values) T.values[r] = c.val;
            if (T.lens) T.lens[r] = c.len;
            if (T.src) T.src[r] = c.src;
          }
        }
        a = v + vlen;
      }
    }
    if (lane == 0)
      for (int t = 0; t < P.n_tags; t++) {
        const TagPlan& T = P.tags[t];
        if (T.valid && ((valid_mask >> t) & 1u)) atomicOr(&T.valid[word], bit);
        if ((seen >> t) & 1u) continue;
        if (T.values) T.values[r] = 0u;
        if (T.lens) T.lens[r] = 0;
        if (T.src) T.src[r] = 0u;
      }
  }
}

// ---------------------------------------------------------------------------------------------
// phase 2: exclusive scans (lengths -> Arrow offsets), all columns in one launch (blockIdx.y = column)
constexpr int SCAN_TPB = 256, SCAN_ITEMS = 8, SCAN_TILE = SCAN_TPB * SCAN_ITEMS;
constexpr int MAX_SCAN_COLS = 6 + MAX_TAGS;

struct ScanCols { int32_t* col[MAX_SCAN_COLS]; int n_cols; uint32_t n; /* elements per column = rows + 1 */ };

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total, uint32_t* ws) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t x = v;
  #pragma unroll
  for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
  if (lane == 31) ws[warp] = x;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < (SCAN_TPB / 32) ? ws[lane] : 0u;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
    ws[lane] = w;
  }
  __syncthreads();
  uint32_t excl = (warp ? ws[warp - 1] : 0u) + x - v;
  *total = ws[SCAN_TPB / 32 - 1];
  __syncthreads();
  return excl;
}

__global__ void __launch_bounds__(SCAN_TPB)
multi_scan_reduce_kernel(ScanCols C, uint64_t* __restrict__ tile_sums, uint32_t n_tiles) {
  __shared__ uint32_t ws[32];
  const int32_t* col = C.col[blockIdx.y];
  uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t s = 0;
  #pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) if (base + k < C.n - 1u) s += (uint32_t)col[base + k];   // element n-1 is the sentinel slot
  uint32_t total;
  block_exclusive_scan(s, &total, ws);
  if (threadIdx.x == 0) tile_sums[(size_t)blockIdx.y * n_tiles + blockIdx.x] = total;
}

// one CTA per column: exclusive scan of the tile sums (64-bit), total -> totals[col]
__global__ void __launch_bounds__(1024)
multi_scan_tiles_kernel(uint64_t* __restrict__ tile_sums, uint32_t n_tiles, uint64_t* __restrict__ totals) {
  __shared__ uint64_t sh[1024];
  __shared__ uint64_t carry;
  uint64_t* ts = tile_sums + (size_t)blockIdx.x * n_tiles;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n_tiles; base += 1024) {
    uint32_t i = base + threadIdx.x;
    uint64_t v = i < n_tiles ? ts[i] : 0ull;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      uint64_t y = threadIdx.x >= (uint32_t)o ? sh[threadIdx.x - o] : 0ull;
      __syncthreads();
      sh[threadIdx.x] += y;
      __syncthreads();
    }
    uint64_t incl = sh[threadIdx.x];
    if (i < n_tiles) ts[i] = carry + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry += incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) totals[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(SCAN_TPB)
multi_scan_apply_kernel(ScanCols C, const uint64_t* __restrict__ tile_sums, uint32_t n_tiles) {
  __shared__ uint32_t ws[32];
  int32_t* col = C.col[blockIdx.y];
  uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS], s = 0;
  #pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) { v[k] = (base + k < C.n - 1u) ? (uint32_t)col[base + k] : 0u; s += v[k]; }
  uint32_t total;
  uint32_t excl = block_exclusive_scan(s, &total, ws);
  uint32_t run = (uint32_t)tile_sums[(size_t)blockIdx.y * n_tiles + blockIdx.x] + excl;
  #pragma unroll
  for (int k = 0; k < SCAN_ITEMS; k++) { if (base + k < C.n) col[base + k] = (int32_t)run; run += v[k]; }
}

// ---------------------------------------------------------------------------------------------
// phase 3: a GROUP of G lanes per record (G = 8 for short reads: four records per warp; G = 32 for long reads)
// out[i] = (in[i] + add) mod 256 (byte-wise, no carry between bytes), 4 bytes per lane and step on destination-aligned
// words; the source word is assembled from two aligned loads.  Returns (per lane) the OR of the "bad byte" masks: an OUTPUT
// byte >= 0x80 (a non-ASCII name byte; a quality q with 95 <= q <= 222, whose char::from(q + 33) is a two-byte UTF-8
// sequence).  The missing-quality fill 0xFF wraps to 0x20 exactly as the reference's u8 addition does in a release build.
// Reads up to 3 bytes past src + n (the inflated buffer carries slack).  `gl` = lane within the group.
template <int G>
__device__ __forceinline__ uint32_t grp_map4(uint8_t* dst, const uint8_t* src, uint32_t n, int gl, uint32_t add4) {
  uint32_t bad = 0;
  const uint32_t add1 = add4 & 0xffu;
  if (n <= (uint32_t)G) {                                      // names, short tags: one predicated byte load / store
    if ((uint32_t)gl < n) { const uint32_t c = (src[gl] + add1) & 0xffu; bad = c & 0x80u; dst[gl] = (uint8_t)c; }
    return bad;
  }
  const uint32_t head = (uint32_t)((4u - (reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u);
  if ((uint32_t)gl < head) { const uint32_t c = (src[gl] + add1) & 0xffu; bad |= c & 0x80u; dst[gl] = (uint8_t)c; }
  dst += head; src += head; n -= head;
  const uint32_t nw = n >> 2;
  const uintptr_t sa = reinterpret_cast<uintptr_t>(src);
  const uint32_t* sw = reinterpret_cast<const uint32_t*>(sa & ~uintptr_t(3));
  const uint32_t sh = (uint32_t)(sa & 3u) * 8u;
  uint32_t* dw = reinterpret_cast<uint32_t*>(dst);
  // four words per lane in flight: the loop is bound by the latency of its loads (ncu: 18 % of the kernel's stall samples sat
  // on the one funnel shift below), not by instruction issue
  for (uint32_t j0 = gl; j0 < nw; j0 += 4 * G) {
    uint32_t lo[4], hi[4];
    #pragma unroll
    for (int k = 0; k < 4; k++) { const uint32_t j = j0 + k * G; const bool in = j < nw; lo[k] = in ? sw[j] : 0u; hi[k] = in ? sw[j + 1] : 0u; }
    #pragma unroll
    for (int k = 0; k < 4; k++) {
      const uint32_t j = j0 + k * G;
      const uint32_t v = __funnelshift_r(lo[k], hi[k], sh);
      const uint32_t o = ((v & 0x7f7f7f7fu) + add4) ^ (v & 0x80808080u);   // per-byte sum mod 256 (add4 bytes are < 0x80)
      if (j < nw) { bad |= o & 0x80808080u; dw[j] = o; }
    }
  }
  const uint32_t t0 = nw << 2;
  if (t0 + (uint32_t)gl < n) { const uint32_t c = (src[t0 + gl] + add1) & 0xffu; bad |= c & 0x80u; dst[t0 + gl] = (uint8_t)c; }
  return bad;
}
template <int G>
__device__ __forceinline__ void grp_copy(uint8_t* dst, const uint8_t* src, uint32_t n, int gl) { (void)grp_map4<G>(dst, src, n, gl, 0u); }

__device__ __forceinline__ uint32_t render_u32(uint8_t* dst, uint32_t v) {   // decimal, returns digits written
  uint32_t d = ndigits_u32(v);
  for (uint32_t k = d; k > 0; k--) { dst[k - 1] = (uint8_t)('0' + v % 10u); v /= 10u; }
  return d;
}
__device__ __forceinline__ uint32_t utf8_put(uint8_t* out, uint32_t cp) {
  if (cp < 0x80u) { out[0] = (uint8_t)cp; return 1; }
  if (cp < 0x800u) { out[0] = 0xC0 | (cp >> 6); out[1] = 0x80 | (cp & 0x3F); return 2; }
  if (cp < 0x10000u) { out[0] = 0xE0 | (cp >> 12); out[1] = 0x80 | ((cp >> 6) & 0x3F); out[2] = 0x80 | (cp & 0x3F); return 3; }
  out[0] = 0xF0 | (cp >> 18); out[1] = 0x80 | ((cp >> 12) & 0x3F); out[2] = 0x80 | ((cp >> 6) & 0x3F); out[3] = 0x80 | (cp & 0x3F);
  return 4;
}

constexpr int VAR_WARPS = 8;
#ifndef BAMSCAN_DV_PREFETCH
#define BAMSCAN_DV_PREFETCH 0          // 1: every column offset of the record is loaded up front (A/B: profiles/r2_decode_var.md)
#endif
#ifndef BAMSCAN_DV_MINBLOCKS
#define BAMSCAN_DV_MINBLOCKS 8
#endif

// One warp instruction serves 32 / G records.  With a warp per 340-byte record (round 1) most steps moved a handful of bytes
// (name 20, chrom 4, CIGAR text 4, MD 3, RG 6) with 32 lanes issued: ~700 warp instructions per record, issue bound at
// 10 % of the HBM roofline.  Eight lanes per record cut that to ~120.  Group-wide shuffles use the width argument; a loop's
// trip count is the maximum over the warp's groups (records of one file are alike, so little is lost).
template <int G>
__global__ void __launch_bounds__(VAR_WARPS * 32, BAMSCAN_DV_MINBLOCKS)
decode_var_kernel(const DecodeParams P) {
  __shared__ uint16_t seq_lut[256];
  {
    const char* codes = "=ACMGRSVTWYHKDBN";
    for (int i = threadIdx.x; i < 256; i += blockDim.x) seq_lut[i] = (uint16_t)((uint8_t)codes[i >> 4] | ((uint16_t)(uint8_t)codes[i & 15] << 8));
  }
  __syncthreads();
  constexpr int GPW = 32 / G;                                  // groups (records) per warp
  const int lane = threadIdx.x & 31, gl = lane & (G - 1);
  const uint8_t* U = P.U;
  // grid-stride over records: a resident warp handles many records, so the LUT set-up and launch cost are amortised.
  // All lanes of a warp run the same number of iterations (shuffles inside): a group past the end works on nothing.
  const uint32_t stride = gridDim.x * VAR_WARPS * GPW;
  for (uint32_t r0 = (blockIdx.x * VAR_WARPS + (threadIdx.x >> 5)) * GPW; r0 < P.n; r0 += stride) {
  const uint32_t r = r0 + (uint32_t)(lane / G);
  const bool on = r < P.n;
  const uint32_t o = on ? P.rec_off[r] : P.rec_off[0];
  const int32_t ref = (int32_t)ld_u32(U, o + 4);
  uint32_t w = ld_u32(U, o + 12);
  const uint32_t l_name = w & 0xffu;
  const uint32_t n_cig = on ? ld_u32(U, o + 16) & 0xffffu : 0u;
  const uint32_t l_seq = on ? ld_u32(U, o + 20) : 0u;
  const int32_t nref = (int32_t)ld_u32(U, o + 24);
  const uint32_t o_name = o + 36, o_cig = o_name + l_name, o_seq = o_cig + 4u * n_cig;
  const uint32_t o_qual = o_seq + (l_seq + 1u) / 2u;
#if BAMSCAN_DV_PREFETCH
  // the per-column output offsets do not depend on the record: loading them here takes one memory round trip off every
  // column's "offset -> bytes -> store" chain (the compiler cannot hoist them itself past the stores below)
  const uint32_t f_name = (P.d_name && on) ? (uint32_t)__ldg(P.l_name + r) : 0u, f_chrom = (P.d_chrom && on) ? (uint32_t)__ldg(P.l_chrom + r) : 0u;
  const uint32_t f_mchrom = (P.d_mchrom && on) ? (uint32_t)__ldg(P.l_mchrom + r) : 0u, f_cigar = (P.d_cigar && on) ? (uint32_t)__ldg(P.l_cigar + r) : 0u;
  const uint32_t f_seq = (P.d_seq && on) ? (uint32_t)__ldg(P.l_seq + r) : 0u, f_qual = (P.d_qual && on) ? (uint32_t)__ldg(P.l_qual + r) : 0u;
#define DV_OFF(col, arr) f_##col
#else
#define DV_OFF(col, arr) (uint32_t)P.arr[r]
#endif

  if (P.d_name && on) {
    uint8_t* dst = P.d_name + DV_OFF(name, l_name);
    uint32_t n = l_name ? l_name - 1u : 0u;
    if (grp_map4<G>(dst, U + o_name, n, gl, 0u)) set_err(P.err, DEC_ERR_NAME, r);
  }
  if (P.d_chrom && on && ref >= 0) grp_copy<G>(P.d_chrom + DV_OFF(chrom, l_chrom), P.ref_names + P.ref_name_off[ref], P.ref_name_off[ref + 1] - P.ref_name_off[ref], gl);
  if (P.d_mchrom && on && nref >= 0) grp_copy<G>(P.d_mchrom + DV_OFF(mchrom, l_mchrom), P.ref_names + P.ref_name_off[nref], P.ref_name_off[nref + 1] - P.ref_name_off[nref], gl);
  if (P.d_cigar) {
    uint8_t* dst = P.d_cigar + (on ? DV_OFF(cigar, l_cigar) : 0u);
    if (P.binary_cigar) { if (on) grp_copy<G>(dst, U + o_cig, 4u * n_cig, gl); }
    else {
      uint32_t base = 0;
      uint32_t nmax = n_cig;                                    // trip count: the largest op count among the warp's groups
      #pragma unroll
      for (int s = G; s < 32; s <<= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, s));
      for (uint32_t k0 = 0; k0 < nmax; k0 += G) {
        uint32_t k = k0 + gl, len = 0, op = 0, wlen = 0;
        if (k < n_cig) { uint32_t cw = ld_u32(U, o_cig + 4u * k); len = cw >> 4; op = cw & 15u; wlen = ndigits_u32(len) + 1u; }
        uint32_t x = wlen;
        #pragma unroll
        for (int s = 1; s < G; s <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, s, G); if (gl >= s) x += y; }
        if (k < n_cig) {
          uint8_t* q = dst + base + x - wlen;
          uint32_t d = render_u32(q, len);
          q[d] = (uint8_t)"MIDNSHP=X"[op > 8u ? 0u : op];
        }
        base += __shfl_sync(0xffffffffu, x, G - 1, G);
      }
    }
  }
  if (P.d_seq && on) {
    uint8_t* dst = P.d_seq + DV_OFF(seq, l_seq);
    // 4 output characters (one aligned word) per lane and step: 2 or 3 input bytes through the two-base LUT
    const uint32_t head = min(l_seq, (uint32_t)((4u - (reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u));
    const uint8_t* ps = U + o_seq;
    if ((uint32_t)gl < head) { uint16_t two = seq_lut[ps[gl >> 1]]; dst[gl] = (uint8_t)((gl & 1) ? (two >> 8) : two); }
    const uint32_t nw = (l_seq - head) >> 2;
    uint32_t* dw = reinterpret_cast<uint32_t*>(dst + head);
    // word j of the output takes the packed bytes 2j, 2j+1 (and the first nibble of 2j+2 when the head was odd); four words per
    // lane in flight (the loads' latency bounds this loop)
    const uint8_t* p2 = ps + (head >> 1);                      // odd head: char `head` is the LOW nibble of p2[0]
    const bool odd = (head & 1u) != 0u;
    for (uint32_t j0 = gl; j0 < nw; j0 += 4 * G) {
      uint32_t b0[4], b1[4], b2[4];
      #pragma unroll
      for (int k = 0; k < 4; k++) {
        const uint32_t j = j0 + k * G; const bool in = j < nw;
        b0[k] = in ? p2[2u * j] : 0u; b1[k] = in ? p2[2u * j + 1u] : 0u; b2[k] = (in && odd) ? p2[2u * j + 2u] : 0u;
      }
      #pragma unroll
      for (int k = 0; k < 4; k++) {
        const uint32_t j = j0 + k * G;
        const uint32_t t0 = seq_lut[b0[k]], t1 = seq_lut[b1[k]], t2 = seq_lut[b2[k]];
        if (j < nw) dw[j] = odd ? ((t0 >> 8) | (t1 << 8) | ((t2 & 0xffu) << 24)) : (t0 | (t1 << 16));
      }
    }
    const uint32_t c0 = head + (nw << 2);
    if (c0 + (uint32_t)gl < l_seq) { const uint32_t c = c0 + gl; uint16_t two = seq_lut[ps[c >> 1]]; dst[c] = (uint8_t)((c & 1u) ? (two >> 8) : two); }
  }
  if (P.d_qual && on && !(P.qual_absent && P.qual_absent[r])) {
    uint8_t* dst = P.d_qual + DV_OFF(qual, l_qual);
    if (grp_map4<G>(dst, U + o_qual, l_seq, gl, 0x21212121u)) set_err(P.err, DEC_ERR_QUAL, r);
  }
  for (int t = 0; t < P.n_tags; t++) {
    const TagPlan& T = P.tags[t];
    if (!T.data || !T.src || !on) continue;
    uint32_t s = T.src[r];
    if (!s) continue;
    const uint8_t ty = U[s];
    const uint32_t v = s + 1u;
    if (T.kind == K_Utf8) {
      uint8_t* dst = T.data + T.lens[r];
      uint32_t n = (uint32_t)(T.lens[r + 1] - T.lens[r]);
      if (ty == 'Z' || ty == 'H') grp_copy<G>(dst, U + v, n, gl);
      else if (gl == 0) {
        if (ty == 'A') utf8_put(dst, U[v]);
        else if (ty == 'f') f32_to_text(ld_u32(U, v), dst);
        else {
          int64_t iv;
          switch (ty) {
            case 'c': iv = (int8_t)U[v]; break;
            case 'C': iv = U[v]; break;
            case 's': iv = (int16_t)ld_u16(U, v); break;
            case 'S': iv = ld_u16(U, v); break;
            case 'i': iv = (int32_t)ld_u32(U, v); break;
            default: iv = ld_u32(U, v); break;
          }
          if (is_scalar_value(iv)) utf8_put(dst, (uint32_t)iv);
          else { if (iv < 0) { *dst++ = '-'; iv = -iv; } render_u32(dst, (uint32_t)iv); }
        }
      }
    } else {   // List<T>: B array, element-wise checked conversion (sam_tag_io.rs:761-1036)
      const uint8_t st = U[v];
      const uint32_t cnt = ld_u32(U, v + 1), es = sub_size(st), e0 = v + 5u;
      const uint32_t first = (uint32_t)T.lens[r];
      const int32_t kind = T.kind;
      bool bad = false;
      for (uint32_t i = gl; i < cnt; i += G) {
        uint32_t a = e0 + i * es;
        int64_t iv = 0; float fv = 0.f; bool isf = false;
        switch (st) {
          case 'c': iv = (int8_t)U[a]; break;
          case 'C': iv = U[a]; break;
          case 's': iv = (int16_t)ld_u16(U, a); break;
          case 'S': iv = ld_u16(U, a); break;
          case 'i': iv = (int32_t)ld_u32(U, a); break;
          case 'I': iv = ld_u32(U, a); break;
          default: fv = __uint_as_float(ld_u32(U, a)); isf = true; break;
        }
        const size_t j = (size_t)first + i;
        switch (kind) {
          case K_ListFloat32: reinterpret_cast<float*>(T.data)[j] = isf ? fv : (st == 'I' ? (float)(uint32_t)iv : (float)(int32_t)iv); break;
          case K_ListInt8: bad |= iv < -128 || iv > 127; reinterpret_cast<int8_t*>(T.data)[j] = (int8_t)iv; break;
          case K_ListUInt8: bad |= iv < 0 || iv > 255; T.data[j] = (uint8_t)iv; break;
          case K_ListInt16: bad |= iv < -32768 || iv > 32767; reinterpret_cast<int16_t*>(T.data)[j] = (int16_t)iv; break;
          case K_ListUInt16: bad |= iv < 0 || iv > 65535; reinterpret_cast<uint16_t*>(T.data)[j] = (uint16_t)iv; break;
          case K_ListInt32: bad |= iv < -2147483648ll || iv > 2147483647ll; reinterpret_cast<int32_t*>(T.data)[j] = (int32_t)iv; break;
          default: bad |= iv < 0; reinterpret_cast<uint32_t*>(T.data)[j] = (uint32_t)iv; break;
        }
      }
      if (bad) set_err(P.err, DEC_ERR_TAG_RANGE, r);
    }
  }
  }
}

}  // namespace bamscan
