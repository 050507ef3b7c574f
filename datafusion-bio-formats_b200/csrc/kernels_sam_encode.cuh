// kernels_sam_encode.cuh -- Arrow columns -> SAM text lines on the device (the SAM write path), sm_100a.
//
// The row rules are the BAM writer's: writer.cu runs enc_cigar_kernel + enc_size_kernel (kernels_encode.cuh) first, unchanged,
// which gives the shared refusals, the resolved reference ids (ref_pairs) and the CIGAR op counts.  Then:
//
//   sam_size_kernel<G>     a GROUP of G lanes per row (G = 8; 32 when the slice averages more than 2 KiB of BAM per row): the
//                          line length and the SAM-only checks (QNAME, SEQ and QUAL alphabets, Z / A characters).  Byte-class
//                          checks run word-wise; CIGAR ops, B elements and scalar tags are spread over the lanes.
//   (exclusive scan of the lengths: dfl::len_tile_sums_kernel / len_offsets_kernel, writer.cu)
//   sam_records_kernel<G>  the same groups write each line at its offset: strings through grp_xform4 (destination-aligned word
//                          stores), CIGAR ops and B elements group-parallel (an element's offset is a group prefix sum of the
//                          text lengths), decimal numbers from registers, floats with f32_to_text (Rust's f32 Display).
//
// Line: QNAME FLAG RNAME POS MAPQ CIGAR RNEXT PNEXT TLEN SEQ QUAL [TG:x:value ...], tab separated, '\n' terminated (DESIGN 3.9).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "f32_text.h"
#include "kernels_encode.cuh"

namespace bamscan {
namespace samenc {

using enc::EncArgs;
using enc::TagCol;

// SAM-only refusals (codes above the shared EncErr values); one code per row, the lowest rule first
enum SamErr : uint32_t {
  SAM_ERR_QNAME = 32, SAM_ERR_SEQ = 33, SAM_ERR_QUAL = 34, SAM_ERR_TAG_Z = 35, SAM_ERR_TAG_A = 36, SAM_ERR_LINE_LEN = 37,
  SAM_ERR_INTERNAL = 38 /* a rendered line does not have its sized length */
};

__device__ __forceinline__ uint32_t dec_len(unsigned long long v) {
  uint32_t n = 1;
  for (unsigned long long p = 10; v >= p && n < 20; p *= 10) n++;
  return n;
}
__device__ __forceinline__ uint32_t sdec_len(long long v) { return v < 0 ? 1u + dec_len(0ull - (unsigned long long)v) : dec_len((unsigned long long)v); }
// writes the n digits of v (n = dec_len(v)) from registers: no global load in the loop
__device__ __forceinline__ void put_dec(uint8_t* out, unsigned long long v, uint32_t n) {
  if (v <= 0xffffffffull) { uint32_t x = (uint32_t)v; for (uint32_t k = n; k-- > 0;) { out[k] = (uint8_t)('0' + x % 10u); x /= 10u; } }
  else { for (uint32_t k = n; k-- > 0;) { out[k] = (uint8_t)('0' + v % 10ull); v /= 10ull; } }
}
__device__ __forceinline__ uint32_t put_sdec(uint8_t* out, long long v) {
  const unsigned long long m = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
  const uint32_t n = dec_len(m);
  if (v < 0) *out++ = '-';
  put_dec(out, m, n);
  return n + (v < 0 ? 1u : 0u);
}

// ---- word-wise byte classes: 0x80 in every byte lane that is OUTSIDE the class ----
__device__ __forceinline__ uint32_t bad_qname(uint32_t v) { return (__vcmpltu4(v, 0x21212121u) | __vcmpgtu4(v, 0x7e7e7e7eu) | __vcmpeq4(v, 0x40404040u)) & 0x80808080u; }  // [!-?A-~]
__device__ __forceinline__ uint32_t bad_seq(uint32_t v) {                                                                                 // [A-Za-z=.]
  const uint32_t l = v | 0x20202020u;
  const uint32_t ok = (__vcmpgeu4(l, 0x61616161u) & __vcmpleu4(l, 0x7a7a7a7au)) | __vcmpeq4(v, 0x3d3d3d3du) | __vcmpeq4(v, 0x2e2e2e2eu);
  return ~ok & 0x80808080u;
}
__device__ __forceinline__ uint32_t bad_qual(uint32_t v) { return __vcmpgtu4(v, 0x7e7e7e7eu) & 0x80808080u; }                              // score > 93
__device__ __forceinline__ uint32_t bad_ztext(uint32_t v) { return (__vcmpltu4(v, 0x20202020u) | __vcmpgtu4(v, 0x7e7e7e7eu)) & 0x80808080u; } // [ !-~]

// OR of cls over src[0 .. n) read by a group: full words with ldw (never past the last byte's word), the tail bytes singly
template <int G, class CLS>
__device__ __forceinline__ uint32_t grp_any4(const uint8_t* src, uint32_t n, int gl, CLS cls) {
  uint32_t bad = 0;
  for (uint32_t j = gl; 4u * j < n; j += G) {
    const uint32_t rem = n - 4u * j;
    const uint8_t* p = src + 4u * j;
    if (rem >= 4) bad |= cls(enc::ldw(p));
    else {
      uint32_t w = 0;
      for (uint32_t k = 0; k < rem; k++) w |= (uint32_t)p[k] << (8u * k);
      bad |= cls(w) & ((1u << (8u * rem)) - 1u);
    }
  }
  return bad;
}

struct OpQualOut { __device__ __forceinline__ uint32_t operator()(uint32_t v) const { return __vmaxu4(v, 0x21212121u); } };   // BAM score max(0, c - 33), + 33
struct OpHexUpper {
  __device__ __forceinline__ uint32_t operator()(uint32_t v) const { return v - ((__vcmpgeu4(v, 0x61616161u) & __vcmpleu4(v, 0x66666666u)) & 0x20202020u); }
};

template <int G>
__device__ __forceinline__ uint32_t grp_incl_scan(uint32_t v, int gl, uint32_t gmask) {
  #pragma unroll
  for (int d = 1; d < G; d <<= 1) { const uint32_t t = __shfl_up_sync(gmask, v, d, G); if (gl >= d) v += t; }
  return v;
}
template <int G>
__device__ __forceinline__ uint32_t grp_or(uint32_t v, uint32_t gmask) {
  #pragma unroll
  for (int o = G / 2; o; o >>= 1) v |= __shfl_xor_sync(gmask, v, o, G);
  return v;
}

// The fixed fields of a row, as every lane of its group sees them.
struct SamRow {
  const uint8_t* name_p; uint32_t name_n;         // name_p == nullptr: '*'
  const uint8_t* rname_p; uint32_t rname_n;       // nullptr: '*'
  const uint8_t* rnext_p; uint32_t rnext_n;       // nullptr: rnext_c
  uint8_t rnext_c;
  uint32_t flag, mapq, pos, pnext; int32_t tlen;
  const uint8_t* cig_p; uint32_t cig_n, n_ops;
  const uint8_t* seq_p; uint32_t l_seq;           // l_seq == 0: '*'
  const uint8_t* qual_p;                          // nullptr: '*'
};

__device__ __forceinline__ uint32_t sam_pos(const enc::PrimCol& c, uint32_t row, bool zero_based) {
  const int64_t r = c.base + row;
  if (!enc::is_valid(c.valid, r)) return 0;
  const unsigned long long p1 = (unsigned long long)c.values[r] + (zero_based ? 1u : 0u);   // (<= 2^31: enc_size_kernel's check)
  return (uint32_t)p1;
}
__device__ __forceinline__ uint32_t prim_or0(const enc::PrimCol& c, uint32_t row) { const int64_t r = c.base + row; return enc::is_valid(c.valid, r) ? c.values[r] : 0u; }

__device__ __forceinline__ SamRow load_row(const EncArgs& a, uint32_t i, uint32_t row, const uint32_t* cig_ops, const int32_t* ref_ids) {
  SamRow s;
  { const int64_t r = a.name.base + row;
    s.name_p = nullptr; s.name_n = 1;
    if (enc::is_valid(a.name.valid, r)) { s.name_p = a.name.data + a.name.off[r]; s.name_n = (uint32_t)(a.name.off[r + 1] - a.name.off[r]); } }
  const int32_t ref = ref_ids[2 * i], mref = ref_ids[2 * i + 1];
  s.rname_p = nullptr; s.rname_n = 1;
  if (ref >= 0) { const int64_t r = a.chrom.base + row; s.rname_p = a.chrom.data + a.chrom.off[r]; s.rname_n = (uint32_t)(a.chrom.off[r + 1] - a.chrom.off[r]); }
  s.rnext_p = nullptr; s.rnext_n = 1; s.rnext_c = '*';
  if (mref >= 0 && mref == ref) s.rnext_c = '=';
  else if (mref >= 0) { const int64_t m = a.mate_chrom.base + row; s.rnext_p = a.mate_chrom.data + a.mate_chrom.off[m]; s.rnext_n = (uint32_t)(a.mate_chrom.off[m + 1] - a.mate_chrom.off[m]); }
  s.flag = prim_or0(a.flags, row); s.mapq = prim_or0(a.mapq, row) & 0xffu; s.tlen = (int32_t)prim_or0(a.tlen, row);
  s.pos = sam_pos(a.start, row, a.zero_based); s.pnext = sam_pos(a.mate_start, row, a.zero_based);
  { const int64_t r = a.cigar.base + row;
    s.cig_p = a.cigar.data + a.cigar.off[r];
    s.cig_n = enc::is_valid(a.cigar.valid, r) ? (uint32_t)(a.cigar.off[r + 1] - a.cigar.off[r]) : 0u;
    s.n_ops = cig_ops[i]; }
  { const int64_t r = a.seq.base + row;
    const uint32_t n = enc::is_valid(a.seq.valid, r) ? (uint32_t)(a.seq.off[r + 1] - a.seq.off[r]) : 0u;
    s.seq_p = a.seq.data + a.seq.off[r];
    s.l_seq = (n == 0 || (n == 1 && s.seq_p[0] == '*')) ? 0u : n;
    const int64_t q = a.qual.base + row;
    const uint32_t qn = enc::is_valid(a.qual.valid, q) ? (uint32_t)(a.qual.off[q + 1] - a.qual.off[q]) : 0u;
    const uint8_t* qp = a.qual.data + a.qual.off[q];
    s.qual_p = (qn == 0 || (qn == 1 && qp[0] == '*')) ? nullptr : qp; }
  return s;
}

// text of the fixed fields without the CIGAR, with the 10 tabs and the '\n'
__device__ __forceinline__ unsigned long long fixed_len(const SamRow& s) {
  return (unsigned long long)s.name_n + dec_len(s.flag) + s.rname_n + dec_len(s.pos) + dec_len(s.mapq) + s.rnext_n + dec_len(s.pnext) +
         sdec_len(s.tlen) + (s.l_seq ? s.l_seq : 1u) + (s.qual_p && s.l_seq ? s.l_seq : 1u) + 11ull;
}

// text length of CIGAR op k (ops are text: the op character at s[k]; binary: word k); 0 for a digit of a text CIGAR
__device__ __forceinline__ uint32_t cigar_op_text(const uint8_t* s, uint32_t k, bool binary, uint32_t* len, uint8_t* opc) {
  if (binary) {
    const uint32_t w = enc::ldw(s + 4u * k);
    *len = w >> 4; *opc = (uint8_t)"MIDNSHP=X"[min(w & 15u, 8u)];
    return dec_len(*len) + 1u;
  }
  const uint8_t c = s[k];
  if (c >= '0' && c <= '9') return 0;
  *len = (uint32_t)enc::digits_before(s, k); *opc = c;
  return dec_len(*len) + 1u;
}

// ---- tags ----
__device__ __forceinline__ bool is_list_kind(int32_t k) { return k >= enc::WK_ListInt8 && k <= enc::WK_ListFloat32; }

// value text of a scalar (non-list) tag that is not a Z / H string; writes it when out != nullptr.  *bad: SAM-only refusal bits.
__device__ __forceinline__ uint32_t scalar_text(const TagCol& t, int64_t r, uint8_t* out, uint32_t* bad) {
  const uint8_t st = t.sam_type;
  if (enc::is_int_kind(t.kind)) {
    bool big;
    const long long v = enc::load_int(t, r, &big);
    if (st == 'A') {
      if (v < 33 || v > 126) *bad |= 16u;
      if (out) out[0] = (uint8_t)v;
      return 1;
    }
    if (out) return put_sdec(out, v);
    return sdec_len(v);
  }
  if (t.kind == enc::WK_Float32 || t.kind == enc::WK_Float64) {
    float f = 0.f;
    if (t.kind == enc::WK_Float32) f = reinterpret_cast<const float*>(t.values)[r];
    else enc::f64_to_f32(reinterpret_cast<const double*>(t.values)[r], &f);   // (out of range: enc_size_kernel refused the row)
    return f32_to_text(__float_as_uint(f), out);
  }
  // Utf8 'A' (one byte: enc_size_kernel's check)
  if (t.off[r + 1] - t.off[r] != 1) { *bad |= 16u; return 1; }
  const uint8_t c = (reinterpret_cast<const uint8_t*>(t.values) + t.off[r])[0];
  if (c < 33 || c > 126) *bad |= 16u;
  if (out) out[0] = c;
  return 1;
}

__device__ __forceinline__ uint32_t list_elem(const TagCol& t, int64_t c, long long* v) {
  switch (t.kind) {
    case enc::WK_ListInt8: *v = reinterpret_cast<const int8_t*>(t.values)[c]; break;
    case enc::WK_ListUInt8: *v = reinterpret_cast<const uint8_t*>(t.values)[c]; break;
    case enc::WK_ListInt16: *v = reinterpret_cast<const int16_t*>(t.values)[c]; break;
    case enc::WK_ListUInt16: *v = reinterpret_cast<const uint16_t*>(t.values)[c]; break;
    case enc::WK_ListInt32: *v = reinterpret_cast<const int32_t*>(t.values)[c]; break;
    case enc::WK_ListUInt32: *v = reinterpret_cast<const uint32_t*>(t.values)[c]; break;
    default: *v = 0; return reinterpret_cast<const uint32_t*>(t.values)[c];       // Float32: the bit pattern
  }
  return 0;
}

// ',' + text of element k of a B field; writes it when out != nullptr.  *range: an integer outside the element type (shared rule).
__device__ __forceinline__ uint32_t list_elem_text(const TagCol& t, int64_t c, uint8_t* out, uint32_t* range) {
  long long v;
  const uint32_t bits = list_elem(t, c, &v);
  if (t.kind == enc::WK_ListFloat32) {
    if (!out) return 1u + f32_to_text(bits, nullptr);
    out[0] = ','; return 1u + f32_to_text(bits, out + 1);
  }
  if (!enc::int_fits(v, t.subtype)) *range = 1;
  if (!out) return 1u + sdec_len(v);
  out[0] = ','; return 1u + put_sdec(out + 1, v);
}

// ---- size pass ----
template <int G>
__global__ void __launch_bounds__(256)
sam_size_kernel(const EncArgs a, const uint32_t* __restrict__ cig_ops, const int32_t* __restrict__ ref_ids, uint32_t* __restrict__ rec_len,
                uint32_t* __restrict__ err) {
  const int lane = threadIdx.x & 31, gl = lane % G;
  const uint32_t i = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (32 / G) + (uint32_t)(lane / G);
  if (i >= a.n_rows) return;                                 // (whole groups: no collective operation reaches a dead lane)
  const uint32_t gmask = G == 32 ? enc::FULLMASK : (((1u << G) - 1u) << (lane - gl));
  const uint32_t row = a.row0 + i;
  const SamRow s = load_row(a, i, row, cig_ops, ref_ids);
  // bits: 1 QNAME, 2 SEQ, 4 QUAL, 8 Z text, 16 A character
  uint32_t bits = 0, range = 0;
  if (s.name_p) {
    if (s.name_n == 0) bits |= 1u;                          // (longer than 254: enc_size_kernel)
    if (grp_any4<G>(s.name_p, s.name_n, gl, bad_qname)) bits |= 1u;
  }
  if (grp_any4<G>(s.seq_p, s.l_seq, gl, bad_seq)) bits |= 2u;
  if (s.qual_p && grp_any4<G>(s.qual_p, s.l_seq, gl, bad_qual)) bits |= 4u;
  unsigned long long part = gl == 0 ? fixed_len(s) : 0ull; // this lane's share of the line
  if (s.n_ops) {
    const bool bin = a.cigar_binary != 0;
    const uint32_t n = bin ? s.cig_n >> 2 : s.cig_n;
    for (uint32_t k = gl; k < n; k += G) { uint32_t len; uint8_t opc; part += cigar_op_text(s.cig_p, k, bin, &len, &opc); }
  } else if (gl == 0) part += 1;                             // '*'
  for (int t = 0; t < a.n_tags; t++) {
    const TagCol& T = a.tags[t];
    const int64_t r = T.base + row;
    if (!enc::is_valid(T.valid, r)) continue;
    if (is_list_kind(T.kind)) {
      const uint32_t b = (uint32_t)T.off[r], n = (uint32_t)T.off[r + 1] - b;
      if (gl == 0) part += 7;                                // \tTG:B:x
      for (uint32_t k = gl; k < n; k += G) part += list_elem_text(T, T.child_base + b + k, nullptr, &range);
    } else if (T.kind == enc::WK_Utf8 && T.sam_type != 'A') {
      const uint32_t b = (uint32_t)T.off[r], n = (uint32_t)T.off[r + 1] - b;
      if (gl == 0) part += 6ull + n;
      if (T.sam_type != 'H' && grp_any4<G>(reinterpret_cast<const uint8_t*>(T.values) + b, n, gl, bad_ztext)) bits |= 8u;
    } else if (t % G == gl) {
      part += 6ull + scalar_text(T, r, nullptr, &bits);
    }
  }
  #pragma unroll
  for (int o = G / 2; o; o >>= 1) part += __shfl_xor_sync(gmask, part, o, G);
  bits = grp_or<G>(bits, gmask);
  range = grp_or<G>(range, gmask);
  if (gl) return;
  unsigned long long total = part;
  if (total > 0x7fffffffull) { bits |= 32u; total = 0; }
  rec_len[i] = (uint32_t)total;
  if (range) enc::report(err, enc::ENC_ERR_TAG_RANGE, row);  // (the BAM writer finds it in its record pass: a shared rule)
  else if (bits) enc::report(err, SAM_ERR_QNAME + (uint32_t)(__ffs((int)bits) - 1), row);
}

// a string field or its '*', then the tab behind it (written by the group's last lane)
template <int G>
__device__ __forceinline__ uint8_t* put_field(uint8_t* p, const uint8_t* src, uint32_t n, uint8_t absent, int gl) {
  if (src) enc::grp_xform4<G>(p, src, n, gl, enc::OpCopy());
  else { if (gl == 0) p[0] = absent; n = 1; }
  if (gl == G - 1) p[n] = '\t';
  return p + n + 1;
}

// ---- record pass ----
template <int G>
__global__ void __launch_bounds__(256)
sam_records_kernel(const EncArgs a, const unsigned long long* __restrict__ rec_off, const uint32_t* __restrict__ cig_ops,
                   const int32_t* __restrict__ ref_ids, uint8_t* __restrict__ out, uint32_t* __restrict__ err) {
  const int lane = threadIdx.x & 31, gl = lane % G;
  const uint32_t i = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (32 / G) + (uint32_t)(lane / G);
  if (i >= a.n_rows) return;
  const uint32_t gmask = G == 32 ? enc::FULLMASK : (((1u << G) - 1u) << (lane - gl));
  const uint32_t row = a.row0 + i;
  const SamRow s = load_row(a, i, row, cig_ops, ref_ids);
  uint8_t* const line = out + rec_off[i];
  uint8_t* const end = out + rec_off[i + 1];
  uint8_t* p = put_field<G>(line, s.name_p, s.name_n, '*', gl);
  // FLAG, RNAME, POS, MAPQ: the numbers go to different lanes
  const uint32_t lf = dec_len(s.flag);
  if (gl == 1 % G) { put_dec(p, s.flag, lf); p[lf] = '\t'; }
  p += lf + 1;
  p = put_field<G>(p, s.rname_p, s.rname_n, '*', gl);
  const uint32_t lp = dec_len(s.pos), lm = dec_len(s.mapq);
  if (gl == 2 % G) { put_dec(p, s.pos, lp); p[lp] = '\t'; }
  if (gl == 3 % G) { put_dec(p + lp + 1, s.mapq, lm); p[lp + 1 + lm] = '\t'; }
  p += lp + 1 + lm + 1;
  // CIGAR: G ops (binary) or G characters (text) per step; an op's offset is the group prefix sum of the op texts before it
  if (s.n_ops) {
    const bool bin = a.cigar_binary != 0;
    const uint32_t n = bin ? s.cig_n >> 2 : s.cig_n;
    uint32_t base = 0;
    for (uint32_t k0 = 0; k0 < n; k0 += G) {
      const uint32_t k = k0 + gl;
      uint32_t len = 0; uint8_t opc = 0;
      const uint32_t tl = k < n ? cigar_op_text(s.cig_p, k, bin, &len, &opc) : 0u;
      const uint32_t incl = grp_incl_scan<G>(tl, gl, gmask);
      if (tl) { uint8_t* q = p + base + incl - tl; put_dec(q, len, tl - 1); q[tl - 1] = opc; }
      base += __shfl_sync(gmask, incl, G - 1, G);
    }
    p += base;
  } else {
    if (gl == 0) p[0] = '*';
    p += 1;
  }
  if (gl == 0) p[0] = '\t';
  p += 1;
  // RNEXT, PNEXT, TLEN
  if (s.rnext_p) p = put_field<G>(p, s.rnext_p, s.rnext_n, '*', gl);
  else p = put_field<G>(p, nullptr, 1, s.rnext_c, gl);
  const uint32_t lq = dec_len(s.pnext), lt = sdec_len(s.tlen);
  if (gl == 4 % G) { put_dec(p, s.pnext, lq); p[lq] = '\t'; }
  if (gl == 5 % G) { put_sdec(p + lq + 1, s.tlen); p[lq + 1 + lt] = '\t'; }
  p += lq + 1 + lt + 1;
  // SEQ (as given), QUAL (score + 33 of the BAM writer's max(0, c - 33))
  if (s.l_seq) enc::grp_xform4<G>(p, s.seq_p, s.l_seq, gl, enc::OpCopy());
  else if (gl == 0) p[0] = '*';
  p += s.l_seq ? s.l_seq : 1u;
  if (gl == 0) p[0] = '\t';
  p += 1;
  if (s.qual_p && s.l_seq) enc::grp_xform4<G>(p, s.qual_p, s.l_seq, gl, OpQualOut());
  else if (gl == 0) p[0] = '*';
  p += (s.qual_p && s.l_seq) ? s.l_seq : 1u;
  // aux fields, tag_fields order: '\t' TG ':' x ':' value
  for (int t = 0; t < a.n_tags; t++) {
    const TagCol& T = a.tags[t];
    const int64_t r = T.base + row;
    if (!enc::is_valid(T.valid, r)) continue;
    const bool list = is_list_kind(T.kind);
    const uint8_t letter = list ? 'B' : (enc::is_int_kind(T.kind) && T.sam_type != 'A') ? 'i' : (T.kind == enc::WK_Float32 || T.kind == enc::WK_Float64) ? 'f' : T.sam_type;
    if (gl == 0) { p[0] = '\t'; p[1] = T.tag[0]; p[2] = T.tag[1]; p[3] = ':'; p[4] = letter; p[5] = ':'; }
    p += 6;
    if (list) {
      const uint32_t b = (uint32_t)T.off[r], n = (uint32_t)T.off[r + 1] - b;
      if (gl == 0) p[0] = T.subtype;
      p += 1;
      const bool flt = T.kind == enc::WK_ListFloat32;
      uint32_t base = 0, range = 0;
      for (uint32_t k0 = 0; k0 < n; k0 += G) {
        const uint32_t k = k0 + gl;
        uint8_t tmp[64];                                     // a float's text is only known once written (<= 1 + 48 bytes)
        const uint32_t tl = k < n ? list_elem_text(T, T.child_base + b + k, flt ? tmp : nullptr, &range) : 0u;
        const uint32_t incl = grp_incl_scan<G>(tl, gl, gmask);
        uint8_t* q = p + base + incl - tl;
        if (tl && flt) { for (uint32_t c = 0; c < tl; c++) q[c] = tmp[c]; }
        else if (tl) list_elem_text(T, T.child_base + b + k, q, &range);
        base += __shfl_sync(gmask, incl, G - 1, G);
      }
      p += base;
    } else if (T.kind == enc::WK_Utf8 && T.sam_type != 'A') {
      const uint32_t b = (uint32_t)T.off[r], n = (uint32_t)T.off[r + 1] - b;
      const uint8_t* src = reinterpret_cast<const uint8_t*>(T.values) + b;
      if (T.sam_type == 'H') enc::grp_xform4<G>(p, src, n, gl, OpHexUpper());
      else enc::grp_xform4<G>(p, src, n, gl, enc::OpCopy());
      p += n;
    } else {
      uint32_t bad = 0, tl = 0;
      if (gl == 0) tl = scalar_text(T, r, p, &bad);
      p += __shfl_sync(gmask, tl, 0, G);
    }
  }
  if (gl == 0) {
    if (p + 1 != end) enc::report(err, SAM_ERR_INTERNAL, row);
    else p[0] = '\n';
  }
}

}  // namespace samenc
}  // namespace bamscan
