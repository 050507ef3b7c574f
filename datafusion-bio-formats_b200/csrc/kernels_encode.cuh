// kernels_encode.cuh -- Arrow columns -> BAM records on the device (SURVEY 8 f4, the write path), sm_100a.
//
// Replaces: batch_to_alignment_records / build_single_record (datafusion/bio-format-core/src/sam_record_serializer.rs:15-212),
// build_tag_data + arrow_to_sam_tag_value (bio-format-core/src/sam_tag_io.rs:109-147, 206-520) and the noodles-bam 0.92.0 record
// encoder behind `writer.write_alignment_record` (bio-format-bam/src/writer.rs:150-166).  Record layout: SAMv1 4.2.
//
//   enc_cigar_kernel    a GROUP of 8 lanes per row: CIGAR op count, reference span, validation (text or binary CIGAR).
//   enc_size_kernel     one THREAD per row: validates the row, resolves chrom / mate_chrom against the header's reference
//                       dictionary (binary search over the sorted names), sizes the aux fields -> record length, reference
//                       ids, n_cigar_op | bin.
//   (exclusive scan of the lengths: writer.cu)
//   enc_records_kernel  a GROUP of G lanes per row (G = 8: four rows per warp): writes the record at its offset in the
//                       uncompressed BAM stream: 36 fixed bytes, name, CIGAR (text parsed group-parallel: an op character's
//                       index is a prefix count of op characters, its length the digits in front of it), 4-bit packed
//                       bases through a shared-memory LUT, qualities - 33 (0xFF when absent), aux fields in tag_fields order.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels_text_common.cuh"

namespace bamscan {
namespace enc {

constexpr int MAX_WTAGS = 32;

enum EncErr : uint32_t {
  ENC_OK = 0, ENC_ERR_FLAGS = 1 /* > 16 bits */, ENC_ERR_CIGAR = 2 /* text does not parse */, ENC_ERR_CIGAR_LEN = 3 /* op length >= 2^28 */,
  ENC_ERR_CIGAR_OPS = 4 /* > 65535 ops (unsupported) */, ENC_ERR_QUAL_LEN = 5, ENC_ERR_NAME_LEN = 6, ENC_ERR_TAG_RANGE = 7, ENC_ERR_TAG_HEX = 8,
  ENC_ERR_TAG_CHAR = 9, ENC_ERR_CIGAR_BIN = 10 /* binary CIGAR: length % 4 or op > 8 */, ENC_ERR_REC_LEN = 11, ENC_ERR_POS = 12 /* position - 1 > i32::MAX */
};

// tag column kinds (== HK_* of bamscan_internal.h)
enum : int32_t { WK_Int8 = 20, WK_UInt8 = 21, WK_Int16 = 22, WK_UInt16 = 23, WK_Int64 = 24, WK_UInt64 = 25, WK_Float64 = 26 };   // scalar tag columns a query may hand over (extract_signed_int / extract_unsigned_int, sam_tag_io.rs:390-438)
enum : int32_t { WK_Int32 = 1, WK_UInt32 = 2, WK_Float32 = 3, WK_Utf8 = 4, WK_ListInt8 = 10, WK_ListUInt8 = 11, WK_ListInt16 = 12,
                 WK_ListUInt16 = 13, WK_ListInt32 = 14, WK_ListUInt32 = 15, WK_ListFloat32 = 16 };

struct Utf8Col { const int32_t* off; const uint8_t* data; const uint8_t* valid; int64_t base; };      // row r -> off[base + r]
struct PrimCol { const uint32_t* values; const uint8_t* valid; int64_t base; };
struct TagCol {
  const void* values;          // Int32 / UInt32 / Float32 values; Utf8: bytes; List: child values
  const int32_t* off;          // Utf8 / List offsets
  const uint8_t* valid;
  int64_t base, child_base;
  int32_t kind;
  uint8_t tag[2], sam_type, subtype;     // subtype: element letter of a 'B' field
};

struct EncArgs {
  Utf8Col name, chrom, cigar, mate_chrom, seq, qual;
  PrimCol start, flags, mapq, mate_start, tlen;
  const uint8_t* ref_blob; const int32_t* ref_off; const int32_t* ref_ids;   // reference names sorted bytewise + their ids
  int32_t n_ref, cigar_binary, zero_based, n_tags;
  uint32_t row0, n_rows;       // this launch covers rows [row0, row0 + n_rows) of the batch
  TagCol tags[MAX_WTAGS];
};

__device__ __forceinline__ bool is_valid(const uint8_t* v, int64_t i) { return !v || ((v[i >> 3] >> (i & 7)) & 1); }

__device__ __forceinline__ int32_t lookup_ref(const EncArgs& a, const uint8_t* s, uint32_t n) { return lookup_ref(a.ref_blob, a.ref_off, a.ref_ids, a.n_ref, s, n); }

__device__ __forceinline__ bool is_int_kind(int32_t k) { return k == WK_Int32 || k == WK_UInt32 || (k >= WK_Int8 && k <= WK_UInt64); }
// the integer at row r of a scalar tag column; *big = a UInt64 beyond i64 (fits no SAM type)
__device__ __forceinline__ long long load_int(const TagCol& t, int64_t r, bool* big) {
  *big = false;
  switch (t.kind) {
    case WK_Int8: return reinterpret_cast<const int8_t*>(t.values)[r];
    case WK_UInt8: return reinterpret_cast<const uint8_t*>(t.values)[r];
    case WK_Int16: return reinterpret_cast<const int16_t*>(t.values)[r];
    case WK_UInt16: return reinterpret_cast<const uint16_t*>(t.values)[r];
    case WK_Int32: return reinterpret_cast<const int32_t*>(t.values)[r];
    case WK_UInt32: return reinterpret_cast<const uint32_t*>(t.values)[r];
    case WK_Int64: return reinterpret_cast<const long long*>(t.values)[r];
    default: { const unsigned long long u = reinterpret_cast<const unsigned long long*>(t.values)[r]; *big = u > 0x7fffffffffffffffull; return (long long)u; }
  }
}
// Float64 -> f32 with the reference's check (finite and within f32's range, sam_tag_io.rs:292-303)
__device__ __forceinline__ bool f64_to_f32(double d, float* out) {
  if (!isfinite(d) || d < -3.4028234663852886e38 || d > 3.4028234663852886e38) return false;
  *out = (float)d;
  return true;
}

// Bytes one aux field occupies in the record (0: NULL / dropped); *e receives a validation error.
__device__ __forceinline__ uint32_t tag_bytes(const TagCol& t, uint32_t row, uint32_t* e) {
  const int64_t r = t.base + row;
  if (!is_valid(t.valid, r)) return 0;
  const uint8_t st = t.sam_type;
  const bool is_int_type = st == 'c' || st == 'C' || st == 's' || st == 'S' || st == 'i' || st == 'I';
  if (is_int_kind(t.kind)) {
    bool big;
    const long long v = load_int(t, r, &big);
    if (is_int_type) { if (big || !int_fits(v, st)) *e = ENC_ERR_TAG_RANGE; return 3u + elem_size(st); }
    if (st == 'A') { if (big || v < 0 || v > 255) *e = ENC_ERR_TAG_CHAR; return 4; }
    *e = ENC_ERR_TAG_RANGE; return 0;                     // (host refuses these combinations before any launch)
  }
  if (t.kind == WK_Float32) return 7;
  if (t.kind == WK_Float64) { float f; if (!f64_to_f32(reinterpret_cast<const double*>(t.values)[r], &f)) *e = ENC_ERR_TAG_RANGE; return 7; }
  if (t.kind == WK_Utf8) {
    const uint32_t b = (uint32_t)t.off[r], n = (uint32_t)t.off[r + 1] - b;
    const uint8_t* s = reinterpret_cast<const uint8_t*>(t.values) + b;
    if (st == 'A') { if (n != 1 || s[0] >= 128) *e = ENC_ERR_TAG_CHAR; return 4; }
    if (st == 'H') {
      bool ok = (n & 1u) == 0;
      for (uint32_t k = 0; k < n && ok; k++) { const uint8_t c = s[k]; ok = (c >= '0' && c <= '9') || (c >= 'A' && c <= 'F') || (c >= 'a' && c <= 'f'); }
      if (!ok) *e = ENC_ERR_TAG_HEX;
    }
    return 3u + n + 1u;
  }
  // lists
  const uint32_t n = (uint32_t)(t.off[r + 1] - t.off[r]);
  return 3u + 1u + 4u + n * elem_size(t.subtype);
}

// CIGAR scan, a group of G lanes per row: op count, reference span (saturating at 2^32 - 1: only `bin` uses it) and validation.
// An op character must follow a digit, its length is the run of digits in front of it, the text must end in an op.  (One thread
// per row walking a 5 000-character long-read CIGAR byte by byte made the size pass 40 x slower than the record writer.)
template <int G>
__global__ void __launch_bounds__(256)
enc_cigar_kernel(const EncArgs a, uint32_t* __restrict__ cig_ops, uint32_t* __restrict__ cig_span, uint32_t* __restrict__ err) {
  const int lane = threadIdx.x & 31, gl = lane % G;
  const uint32_t i = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (32 / G) + (uint32_t)(lane / G);
  const bool live = i < a.n_rows;
  const uint32_t row = a.row0 + (live ? i : 0u);
  const int64_t r = a.cigar.base + row;
  const uint8_t* s = a.cigar.data + a.cigar.off[r];
  const uint32_t n = (live && is_valid(a.cigar.valid, r)) ? (uint32_t)(a.cigar.off[r + 1] - a.cigar.off[r]) : 0u;
  uint32_t ops = 0, e = ENC_OK; unsigned long long span = 0;
  if (a.cigar_binary) {
    if (n & 3u) e = ENC_ERR_CIGAR_BIN;
    for (uint32_t k = gl; k < (n >> 2); k += G) {
      const uint32_t w = (uint32_t)s[4 * k] | ((uint32_t)s[4 * k + 1] << 8) | ((uint32_t)s[4 * k + 2] << 16) | ((uint32_t)s[4 * k + 3] << 24);
      const uint32_t op = w & 15u;
      if (op > 8u) e = ENC_ERR_CIGAR_BIN;
      if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += w >> 4;
      ops++;
    }
  } else if (!(n == 0 || (n == 1 && s[0] == '*'))) {
    for (uint32_t k = gl; k < n; k += G) {
      const uint8_t c = s[k];
      if (c >= '0' && c <= '9') continue;
      const int op = op_code(c);
      if (op < 0 || k == 0 || s[k - 1] < '0' || s[k - 1] > '9') e = ENC_ERR_CIGAR;
      const unsigned long long len = digits_before(s, k);
      if (len >= (1ull << 28)) e = ENC_ERR_CIGAR_LEN;
      else if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += len;
      ops++;
    }
    if (gl == 0 && s[n - 1] >= '0' && s[n - 1] <= '9') e = ENC_ERR_CIGAR;
  }
  #pragma unroll
  for (int o = G / 2; o; o >>= 1) {
    ops += __shfl_xor_sync(FULLMASK, ops, o, G);
    span += __shfl_xor_sync(FULLMASK, span, o, G);
    e = max(e, __shfl_xor_sync(FULLMASK, e, o, G));
  }
  if (!live || gl) return;
  if (ops > 65535u) e = ENC_ERR_CIGAR_OPS;
  cig_ops[i] = ops; cig_span[i] = (uint32_t)min(span, 0xffffffffull);
  if (e) report(err, e, row);
}

__global__ void __launch_bounds__(256)
enc_size_kernel(const EncArgs a, const uint32_t* __restrict__ cig_ops, const uint32_t* __restrict__ cig_span, uint32_t* __restrict__ rec_len,
                int32_t* __restrict__ ref_ids, uint32_t* __restrict__ cig_bin, uint32_t* __restrict__ err) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n_rows) return;
  const uint32_t row = a.row0 + i;
  uint32_t e = ENC_OK;
  // name: NULL or "*" -> "*" (sam_record_serializer.rs:116-121 + the encoder's missing-name rule)
  uint32_t l_name = 1;
  {
    const int64_t r = a.name.base + row;
    if (is_valid(a.name.valid, r)) l_name = (uint32_t)(a.name.off[r + 1] - a.name.off[r]);      // ("*" is written as it stands; an empty name stays empty)
    if (l_name > 254) e = ENC_ERR_NAME_LEN;
  }
  if (a.flags.values[a.flags.base + row] > 0xffffu) e = ENC_ERR_FLAGS;
  int32_t ref = -1, mref = -1;
  {
    const int64_t r = a.chrom.base + row;
    if (is_valid(a.chrom.valid, r)) ref = lookup_ref(a, a.chrom.data + a.chrom.off[r], (uint32_t)(a.chrom.off[r + 1] - a.chrom.off[r]));
    const int64_t m = a.mate_chrom.base + row;
    if (is_valid(a.mate_chrom.valid, m)) {
      const uint8_t* s = a.mate_chrom.data + a.mate_chrom.off[m];
      const uint32_t n = (uint32_t)(a.mate_chrom.off[m + 1] - a.mate_chrom.off[m]);
      mref = (n == 1 && s[0] == '=') ? ref : lookup_ref(a, s, n);
    }
  }
  // CIGAR: op count + reference span come from enc_cigar_kernel
  const uint32_t n_ops = cig_ops[i]; const unsigned long long span = cig_span[i];
  // sequence / qualities ("*" and "" are absent)
  uint32_t l_seq = 0;
  {
    const int64_t r = a.seq.base + row;
    const uint32_t n = is_valid(a.seq.valid, r) ? (uint32_t)(a.seq.off[r + 1] - a.seq.off[r]) : 0u;
    if (!(n == 0 || (n == 1 && a.seq.data[a.seq.off[r]] == '*'))) l_seq = n;
    const int64_t q = a.qual.base + row;
    const uint32_t qn = is_valid(a.qual.valid, q) ? (uint32_t)(a.qual.off[q + 1] - a.qual.off[q]) : 0u;
    const bool q_absent = qn == 0 || (qn == 1 && a.qual.data[a.qual.off[q]] == '*');
    if (!q_absent && qn != l_seq) e = ENC_ERR_QUAL_LEN;
  }
  {
    const int64_t m = a.mate_start.base + row;      // the encoder's i32::try_from(position - 1)
    if (is_valid(a.mate_start.valid, m) && (unsigned long long)a.mate_start.values[m] + (a.zero_based ? 1u : 0u) > 0x80000000ull) e = ENC_ERR_POS;
  }
  // bin (RecordBuf::alignment_end is start + span - 1, unconditionally; Position 0 does not exist -> the unmapped bin)
  uint32_t bin = 4680;
  {
    const int64_t r = a.start.base + row;
    if (is_valid(a.start.valid, r)) {
      const unsigned long long p1 = (unsigned long long)a.start.values[r] + (a.zero_based ? 1u : 0u);
      if (p1 > 0x80000000ull) e = ENC_ERR_POS;
      if (p1 >= 1) {
        const unsigned long long end1 = p1 + span - 1;
        if (end1 >= 1) {
          const unsigned long long s0 = p1 - 1, e0 = end1 - 1;
          if (s0 >> 14 == e0 >> 14) bin = 4681 + (uint32_t)(s0 >> 14);
          else if (s0 >> 17 == e0 >> 17) bin = 585 + (uint32_t)(s0 >> 17);
          else if (s0 >> 20 == e0 >> 20) bin = 73 + (uint32_t)(s0 >> 20);
          else if (s0 >> 23 == e0 >> 23) bin = 9 + (uint32_t)(s0 >> 23);
          else if (s0 >> 26 == e0 >> 26) bin = 1 + (uint32_t)(s0 >> 26);
          else bin = 0;
        }
      }
    }
  }
  unsigned long long total = 4ull + 32ull + l_name + 1ull + 4ull * n_ops + (l_seq + 1u) / 2u + l_seq;
  for (int t = 0; t < a.n_tags; t++) total += tag_bytes(a.tags[t], row, &e);
  if (total > 0x7fffffffull) { e = ENC_ERR_REC_LEN; total = 36; }
  rec_len[i] = (uint32_t)total;
  ref_ids[2 * i] = ref; ref_ids[2 * i + 1] = mref;
  cig_bin[i] = n_ops | ((bin & 0xffffu) << 16);
  if (e) report(err, e, row);
}

// ---- record writer ----
template <int G>
__global__ void __launch_bounds__(256)
enc_records_kernel(const EncArgs a, const unsigned long long* __restrict__ rec_off, const int32_t* __restrict__ ref_ids,
                   const uint32_t* __restrict__ cig_bin, uint8_t* __restrict__ out, uint32_t* __restrict__ err) {
  __shared__ uint8_t base_code[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    const char* B = "=ACMGRSVTWYHKDBN";
    uint8_t c = 15;
    #pragma unroll
    for (int k = 0; k < 16; k++) if (i == B[k] || (i >= 'a' && i <= 'z' && i - 32 == B[k])) c = (uint8_t)k;
    base_code[i] = c;
  }
  __syncthreads();
  constexpr int RPW = 32 / G;
  const int lane = threadIdx.x & 31, gl = lane % G, gbase = lane - gl;
  const uint32_t gmask = G == 32 ? FULLMASK : (((1u << G) - 1u) << gbase);
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t i = warp * RPW + (uint32_t)(lane / G);
  const bool live = i < a.n_rows;
  const uint32_t row = a.row0 + (live ? i : 0u);
  uint8_t* const rec = out + (live ? rec_off[i] : 0ull);
  const uint32_t total = live ? (uint32_t)(rec_off[i + 1] - rec_off[i]) : 0u;
  // ---- geometry (every lane of the group computes the same values) ----
  uint32_t l_name = 1, name_n = 0; const uint8_t* name_p = nullptr;
  uint32_t l_seq = 0; const uint8_t* seq_p = nullptr; const uint8_t* qual_p = nullptr;
  uint32_t cig_n = 0; const uint8_t* cig_p = nullptr; uint32_t n_ops = 0, bin = 4680;
  if (live) {
    { const int64_t r = a.name.base + row;
      if (is_valid(a.name.valid, r)) { name_n = (uint32_t)(a.name.off[r + 1] - a.name.off[r]); name_p = a.name.data + a.name.off[r]; l_name = name_n; } }
    { const int64_t r = a.seq.base + row;
      const uint32_t n = is_valid(a.seq.valid, r) ? (uint32_t)(a.seq.off[r + 1] - a.seq.off[r]) : 0u;
      seq_p = a.seq.data + a.seq.off[r];
      if (!(n == 0 || (n == 1 && seq_p[0] == '*'))) l_seq = n;
      const int64_t q = a.qual.base + row;
      const uint32_t qn = is_valid(a.qual.valid, q) ? (uint32_t)(a.qual.off[q + 1] - a.qual.off[q]) : 0u;
      const uint8_t* qp = a.qual.data + a.qual.off[q];
      if (!(qn == 0 || (qn == 1 && qp[0] == '*'))) qual_p = qp; }
    { const int64_t r = a.cigar.base + row;
      cig_p = a.cigar.data + a.cigar.off[r];
      cig_n = is_valid(a.cigar.valid, r) ? (uint32_t)(a.cigar.off[r + 1] - a.cigar.off[r]) : 0u;
      if (!a.cigar_binary && cig_n == 1 && cig_p[0] == '*') cig_n = 0; }
    n_ops = cig_bin[i] & 0xffffu; bin = cig_bin[i] >> 16;
  }
  // ---- 36 fixed bytes: nine words, lane j of the group writes word j (lane 0 also word 8) ----
  if (live) {
    uint32_t w[9];
    w[0] = total - 4u;
    w[1] = (uint32_t)ref_ids[2 * i];
    { const int64_t r = a.start.base + row;
      const unsigned long long p1 = is_valid(a.start.valid, r) ? (unsigned long long)a.start.values[r] + (a.zero_based ? 1u : 0u) : 0ull;
      w[2] = p1 >= 1 ? (uint32_t)(p1 - 1) : 0xffffffffu; }
    w[3] = (l_name + 1u) | ((a.mapq.values[a.mapq.base + row] & 0xffu) << 8) | (bin << 16);
    w[4] = n_ops | ((a.flags.values[a.flags.base + row] & 0xffffu) << 16);
    w[5] = l_seq;
    w[6] = (uint32_t)ref_ids[2 * i + 1];
    { const int64_t r = a.mate_start.base + row;
      const unsigned long long p1 = is_valid(a.mate_start.valid, r) ? (unsigned long long)a.mate_start.values[r] + (a.zero_based ? 1u : 0u) : 0ull;
      w[7] = p1 >= 1 ? (uint32_t)(p1 - 1) : 0xffffffffu; }
    w[8] = a.tlen.values[a.tlen.base + row];
    {
      // 36 bytes at an arbitrary byte offset: the aligned words inside them are funnel shifts of two neighbouring header words,
      // the 0..3 bytes in front of the first and behind the last aligned word go singly
      const uint32_t al = (uint32_t)(reinterpret_cast<uintptr_t>(rec) & 3u);
      if (al == 0) {
        #pragma unroll
        for (int j = 0; j < 9; j++) if (j % G == gl) reinterpret_cast<uint32_t*>(rec)[j] = w[j];
      } else {
        const uint32_t hb = 4u - al;                         // bytes of w[0] in front of the first aligned word
        if ((uint32_t)gl < hb) rec[gl] = (uint8_t)(w[0] >> (8u * gl));
        uint32_t* aw = reinterpret_cast<uint32_t*>(rec + hb);
        #pragma unroll
        for (int j = 0; j < 8; j++) if (j % G == gl) aw[j] = __funnelshift_r(w[j], w[j + 1], hb * 8u);
        if ((uint32_t)gl < al) rec[hb + 32u + gl] = (uint8_t)(w[8] >> (8u * (hb + gl)));
      }
    }
    // ---- name + NUL ----
    uint8_t* np = rec + 36;
    if (name_p) grp_xform4<G>(np, name_p, name_n, gl, OpCopy());
    else if (gl == 0) np[0] = '*';
    if (gl == 0) np[l_name] = 0;
  }
  uint8_t* const cp = rec + 36 + l_name + 1;
  // ---- CIGAR ----
  if (a.cigar_binary) {
    if (live) for (uint32_t k = gl; k < cig_n; k += G) cp[k] = cig_p[k];
  } else {
    // text: G characters per step; an op character's index is the number of op characters in front of it
    uint32_t steps = (cig_n + G - 1) / G;
    #pragma unroll
    for (int o = 16; o; o >>= 1) steps = max(steps, __shfl_xor_sync(FULLMASK, steps, o));     // warp-uniform trip count (ballots below)
    uint32_t ops_before = 0;
    for (uint32_t s = 0; s < steps; s++) {
      const uint32_t k = s * G + gl;
      const uint8_t c = (live && k < cig_n) ? cig_p[k] : (uint8_t)'0';
      const bool is_op = !(c >= '0' && c <= '9');
      const uint32_t bal = (__ballot_sync(FULLMASK, is_op) & gmask) >> gbase;
      if (is_op) {
        const uint32_t len = (uint32_t)digits_before(cig_p, k);
        const uint32_t idx = ops_before + __popc(bal & ((1u << gl) - 1u));
        if (idx < n_ops) st_u32(cp + 4 * idx, (len << 4) | (uint32_t)max(op_code(c), 0));
      }
      ops_before += __popc(bal);
    }
  }
  if (!live) return;
  // ---- bases (two per byte, high nibble first) + qualities ----
  uint8_t* const sp = cp + 4 * n_ops;
  const uint32_t nb = (l_seq + 1u) >> 1;
  {
    // packed byte k holds bases 2k (high nibble) and 2k + 1; one aligned output word = 8 bases = two unaligned source words
    auto pack1 = [&](uint32_t k) { const uint32_t hi = base_code[seq_p[2 * k]], lo = (2 * k + 1 < l_seq) ? base_code[seq_p[2 * k + 1]] : 0u; return (uint8_t)((hi << 4) | lo); };
    const uint32_t full = l_seq >> 1;                        // packed bytes made of two real bases
    const uint32_t head = min(full, (uint32_t)((4u - (reinterpret_cast<uintptr_t>(sp) & 3u)) & 3u));
    if ((uint32_t)gl < head) sp[gl] = pack1(gl);
    const uint32_t nw = (full - head) >> 2;
    uint32_t* dw = reinterpret_cast<uint32_t*>(sp + head);
    const uint8_t* s8 = seq_p + 2u * head;
    for (uint32_t j = gl; j < nw; j += G) {
      const uint32_t x = ldw(s8 + 8u * j), y = ldw(s8 + 8u * j + 4u);
      const uint32_t b0 = (base_code[x & 0xffu] << 4) | base_code[(x >> 8) & 0xffu], b1 = (base_code[(x >> 16) & 0xffu] << 4) | base_code[x >> 24];
      const uint32_t b2 = (base_code[y & 0xffu] << 4) | base_code[(y >> 8) & 0xffu], b3 = (base_code[(y >> 16) & 0xffu] << 4) | base_code[y >> 24];
      dw[j] = b0 | (b1 << 8) | (b2 << 16) | (b3 << 24);
    }
    const uint32_t t0 = head + (nw << 2);
    if (t0 + (uint32_t)gl < nb) sp[t0 + gl] = pack1(t0 + gl);  // <= 3 full bytes + the odd last base
  }
  uint8_t* const qp = sp + nb;
  if (qual_p) grp_xform4<G>(qp, qual_p, l_seq, gl, OpQual());
  else { for (uint32_t k = gl; k < l_seq; k += G) qp[k] = 0xff; }
  // ---- aux fields, tag_fields order ----
  uint8_t* ap = qp + l_seq;
  for (int t = 0; t < a.n_tags; t++) {
    const TagCol& T = a.tags[t];
    uint32_t e = 0;
    const uint32_t nbytes = tag_bytes(T, row, &e);
    if (!nbytes) continue;
    const int64_t r = T.base + row;
    const uint8_t st = T.sam_type;
    if (gl == 0) { ap[0] = T.tag[0]; ap[1] = T.tag[1]; }
    if (is_int_kind(T.kind)) {
      bool big;
      const uint32_t v = (uint32_t)load_int(T, r, &big);
      if (gl == 0) { ap[2] = st; const uint32_t es = st == 'A' ? 1u : elem_size(st); ap[3] = (uint8_t)v; if (es > 1) ap[4] = (uint8_t)(v >> 8); if (es > 2) { ap[5] = (uint8_t)(v >> 16); ap[6] = (uint8_t)(v >> 24); } }
    } else if (T.kind == WK_Float32) {
      if (gl == 0) { ap[2] = 'f'; st_u32(ap + 3, reinterpret_cast<const uint32_t*>(T.values)[r]); }
    } else if (T.kind == WK_Float64) {
      float f = 0.f; f64_to_f32(reinterpret_cast<const double*>(T.values)[r], &f);
      if (gl == 0) { ap[2] = 'f'; st_u32(ap + 3, __float_as_uint(f)); }
    } else if (T.kind == WK_Utf8) {
      const uint32_t b = (uint32_t)T.off[r], n = (uint32_t)T.off[r + 1] - b;
      const uint8_t* s = reinterpret_cast<const uint8_t*>(T.values) + b;
      if (st == 'A') { if (gl == 0) { ap[2] = 'A'; ap[3] = s[0]; } }
      else {
        if (gl == 0) { ap[2] = st == 'H' ? 'H' : 'Z'; ap[3 + n] = 0; }
        if (st == 'H') { for (uint32_t k = gl; k < n; k += G) { uint8_t c = s[k]; if (c >= 'a' && c <= 'f') c -= 32; ap[3 + k] = c; } }
        else grp_xform4<G>(ap + 3, s, n, gl, OpCopy());
      }
    } else {
      const uint32_t b = (uint32_t)T.off[r], n = (uint32_t)T.off[r + 1] - b;
      const uint8_t sub = T.subtype;
      const uint32_t es = elem_size(sub);
      if (gl == 0) { ap[2] = 'B'; ap[3] = sub; st_u32(ap + 4, n); }
      uint8_t* ep = ap + 8;
      const int64_t c0 = T.child_base + b;
      for (uint32_t k = gl; k < n; k += G) {
        long long v; uint32_t raw;
        switch (T.kind) {
          case WK_ListInt8: v = reinterpret_cast<const int8_t*>(T.values)[c0 + k]; break;
          case WK_ListUInt8: v = reinterpret_cast<const uint8_t*>(T.values)[c0 + k]; break;
          case WK_ListInt16: v = reinterpret_cast<const int16_t*>(T.values)[c0 + k]; break;
          case WK_ListUInt16: v = reinterpret_cast<const uint16_t*>(T.values)[c0 + k]; break;
          case WK_ListInt32: v = reinterpret_cast<const int32_t*>(T.values)[c0 + k]; break;
          case WK_ListUInt32: v = reinterpret_cast<const uint32_t*>(T.values)[c0 + k]; break;
          default: v = 0; break;
        }
        if (T.kind == WK_ListFloat32) raw = reinterpret_cast<const uint32_t*>(T.values)[c0 + k];
        else { raw = (uint32_t)v; if (!int_fits(v, sub)) report(err, ENC_ERR_TAG_RANGE, row); }
        if (es == 1) ep[k] = (uint8_t)raw; else if (es == 2) st_u16(ep + 2 * k, raw); else st_u32(ep + 4 * k, raw);
      }
    }
    ap += nbytes;
  }
}

}  // namespace enc
}  // namespace bamscan
